//! Drop-in batch entry points for looping over `elastic_elgamal`'s per-item calls (Ristretto backend).
//!
//! ```ignore
//! // before (examples/voting.rs:189-204):
//! for ballot in &ballots { let cts = ballot.verify(&params)?; for (t, c) in totals.iter_mut().zip(cts) { *t += *c; } }
//! // after: all GPUs of the box, tally combined inside the library (one ncclAllGather + a point-addition kernel)
//! let engine = Engine::new_multi(&[0, 1, 2, 3, 4, 5, 6, 7])?;
//! engine.set_receiver(params.receiver())?;
//! let outcome = engine.verify_choices(&params, &ballots)?;   // outcome.verdicts[i], outcome.tally
//! ```
//!
//! Every method is `items.iter().map(|x| x.verify(..))` (or `::new(..)`) over a batch, with the reference's own result and
//! error types per item.  Objects travel as the flat byte layouts of `include/eg_b200.h`: `to_bytes` where the reference
//! has one, otherwise their binary serde form with everything but the byte fields dropped (`flat`).
//!
//! Source only in the build image (no rustc there); `tests/test_c_abi.py` keeps the `-sys` declarations in step with the
//! header.  See INTEGRATION.md for the mapping onto the reference's types.

pub mod flat;

use elastic_elgamal::{
    app::{
        ChoiceParams, ChoiceVerificationError, EncryptedChoice, MultiChoice, QuadraticVotingBallot, QuadraticVotingError,
        QuadraticVotingParams, SingleChoice,
    },
    group::{ElementOps, Ristretto, ScalarOps},
    sharing::{self, PublicKeySet},
    CandidateDecryption, Ciphertext, CommitmentEquivalenceProof, LogEqualityProof, ProofOfPossession, PublicKey,
    RangeDecomposition, RangeProof, RingProof, SecretKey, SumOfSquaresProof, VerifiableDecryption, VerificationError,
};
use elastic_elgamal_b200_sys as sys;
use serde::Serialize;
use std::{
    ffi::{CStr, CString},
    ptr,
};

type Element = <Ristretto as ElementOps>::Element;
type Scalar = <Ristretto as ScalarOps>::Scalar;

/// API / CUDA / NCCL failures (never a per-item outcome).
#[derive(Debug)]
pub struct EngineError {
    pub status: sys::eg_status,
    pub message: String,
}

impl std::fmt::Display for EngineError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "eg_b200 status {}: {}", self.status, self.message)
    }
}
impl std::error::Error for EngineError {}

impl From<flat::FlatError> for EngineError {
    fn from(e: flat::FlatError) -> Self {
        EngineError { status: sys::EG_ERR_INVALID_ARG, message: e.0 }
    }
}

/// Why a tally of [`Engine::combine_accepted_and_decrypt`] has no decryption.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum CombineError {
    /// Fewer than `threshold` of the tally's shares were accepted: `Params::combine_shares` returns `None`.
    NotEnoughShares,
}

/// One context: a single GPU (`new`), all chosen GPUs of the box (`new_multi`), or one rank of a multi-process job
/// (`new` + `attach_comm`).  `!Sync`: use from one thread at a time; independent across instances.
pub struct Engine {
    ctx: *mut sys::eg_ctx,
}

unsafe impl Send for Engine {}

/// Where a prover takes its randomness from.
pub enum Randomness<'a> {
    /// 64-byte blocks in the reference's draw order (one per `generate_scalar` call), `draws * 64` bytes per item.
    Blocks(&'a [u8]),
    /// In-kernel ChaCha20 (`rand_chacha::ChaCha20Rng` semantics): item `i` draws blocks `counter_base + (i << 20) + k`.
    Seeded { seed: &'a [u8; 32], counter_base: u64 },
}

pub struct ChoiceOutcome {
    /// `Ok(())` or the error `EncryptedChoice::verify` would have returned, per ballot.
    pub verdicts: Vec<Result<(), ChoiceVerificationError>>,
    /// Sum of the verified ballots' ciphertexts, one per option (over all GPUs / ranks of the context).
    pub tally: Vec<Ciphertext<Ristretto>>,
}

pub struct QvOutcome {
    pub verdicts: Vec<Result<(), QuadraticVotingError>>,
    pub tally: Vec<Ciphertext<Ristretto>>,
}

/// `DiscreteLogTable::new(lo..hi)` resident on the engine's device(s).
pub struct DlogTable<'e> {
    engine: &'e Engine,
    table: *mut sys::eg_dlog_table,
}

impl DlogTable<'_> {
    /// `DiscreteLogTable::get` (encryption.rs:287-297) over a batch of elements: `Some(value)` when the element is `[value]G`
    /// with `value` in the table's range (the identity is `Some(0)`), else `None`.
    pub fn get_batch(&self, elements: &[<Ristretto as elastic_elgamal::group::ElementOps>::Element]) -> Result<Vec<Option<u64>>, EngineError> {
        let n = elements.len();
        let mut bytes = vec![0_u8; 32 * n];
        for (el, chunk) in elements.iter().zip(bytes.chunks_mut(32)) {
            Ristretto::serialize_element(el, chunk);
        }
        let (mut values, mut found) = (vec![0_u64; n], vec![0_u8; n]);
        self.engine.check(unsafe {
            sys::eg_dlog_lookup_batch(self.engine.ctx, self.table, n, bytes.as_ptr(), values.as_mut_ptr(), found.as_mut_ptr())
        })?;
        Ok(values.iter().zip(found).map(|(&v, f)| (f == 1).then_some(v)).collect())
    }
}

impl Drop for DlogTable<'_> {
    fn drop(&mut self) {
        let _ = self.engine;
        unsafe { sys::eg_dlog_table_destroy(self.table) }
    }
}

fn element(bytes: &[u8]) -> Element {
    Ristretto::deserialize_element(bytes).expect("the engine emits canonical encodings")
}

fn ciphertexts(bytes: &[u8]) -> Vec<Ciphertext<Ristretto>> {
    bytes.chunks(64).map(|c| Ciphertext::from_elements(element(&c[..32]), element(&c[32..]))).collect()
}

/// `VerificationError` of a plain proof verdict byte; malformed encodings cannot reach `verify` through typed inputs.
fn proof_verdict(v: u8) -> Result<(), VerificationError> {
    if v == sys::EG_V_OK { Ok(()) } else { Err(VerificationError::ChallengeMismatch) }
}

fn range_spec(decomposition: &RangeDecomposition) -> Result<sys::eg_range, EngineError> {
    // `RangeDecomposition` exposes its rings only through `Display` ("6 * 0..3 + 2 * 0..3 + 0..2", range.rs:110-124)
    let mut spec = sys::eg_range { n_rings: 0, reserved: 0, size: [0; 64], step: [0; 64] };
    for (i, term) in decomposition.to_string().split(" + ").enumerate() {
        let (step, range) = match term.split_once(" * ") {
            Some((step, range)) => (step.parse::<u64>().ok(), range),
            None => (Some(1), term),
        };
        let size = range.strip_prefix("0..").and_then(|s| s.parse::<u64>().ok());
        match (step, size, i < 64) {
            (Some(step), Some(size), true) => {
                spec.step[i] = step;
                spec.size[i] = size;
                spec.n_rings = i as u32 + 1;
            }
            _ => return Err(EngineError { status: sys::EG_ERR_INVALID_ARG, message: format!("cannot parse range decomposition `{decomposition}`") }),
        }
    }
    Ok(spec)
}

impl Engine {
    /// One GPU.
    pub fn new(device: i32) -> Result<Self, EngineError> {
        let mut ctx = ptr::null_mut();
        let status = unsafe { sys::eg_ctx_create(device, &mut ctx) };
        if status != sys::EG_SUCCESS {
            return Err(EngineError { status, message: "eg_ctx_create failed (no CUDA device? there is no CPU fallback)".into() });
        }
        Ok(Self { ctx })
    }

    /// Several GPUs driven from this process: batches shard across them, tallies are combined inside the library.
    pub fn new_multi(devices: &[i32]) -> Result<Self, EngineError> {
        let mut ctx = ptr::null_mut();
        let status = unsafe { sys::eg_ctx_create_multi(devices.as_ptr(), devices.len() as i32, &mut ctx) };
        if status != sys::EG_SUCCESS {
            return Err(EngineError { status, message: "eg_ctx_create_multi failed (devices / libnccl.so.2?)".into() });
        }
        Ok(Self { ctx })
    }

    /// Rank 0 of a multi-process job creates the id; the host sends its 128 bytes to the other ranks.
    pub fn comm_unique_id() -> Result<[u8; sys::EG_COMM_ID_BYTES], EngineError> {
        let mut id = [0_u8; sys::EG_COMM_ID_BYTES];
        let status = unsafe { sys::eg_comm_unique_id(id.as_mut_ptr()) };
        if status == sys::EG_SUCCESS { Ok(id) } else { Err(EngineError { status, message: "libnccl.so.2 could not be loaded".into() }) }
    }

    /// Collective: every rank calls it once.  Afterwards `verify_choices` / `verify_qv_ballots` are collective and their
    /// tallies are the totals over all ranks.
    pub fn attach_comm(&self, id: &[u8; sys::EG_COMM_ID_BYTES], rank: i32, world: i32) -> Result<(), EngineError> {
        self.check(unsafe { sys::eg_ctx_attach_comm(self.ctx, id.as_ptr(), rank, world) })
    }

    fn check(&self, status: sys::eg_status) -> Result<(), EngineError> {
        if status == sys::EG_SUCCESS {
            return Ok(());
        }
        let message = unsafe { CStr::from_ptr(sys::eg_last_error(self.ctx)) }.to_string_lossy().into_owned();
        Err(EngineError { status, message })
    }

    /// Mirrors `PublicKey::from_bytes` validation and builds the key's fixed-base table.
    pub fn set_receiver(&self, key: &PublicKey<Ristretto>) -> Result<(), EngineError> {
        self.check(unsafe { sys::eg_ctx_set_receiver(self.ctx, key.as_bytes().as_ptr()) })
    }

    /// The Pedersen blinding base of `CommitmentEquivalenceProof` (`commitment_blinding_base`).
    pub fn set_blinding_base(&self, base: &Element) -> Result<(), EngineError> {
        let mut bytes = [0_u8; 32];
        Ristretto::serialize_element(base, &mut bytes);
        self.check(unsafe { sys::eg_ctx_set_blinding_base(self.ctx, bytes.as_ptr()) })
    }

    /// `true`: constant-time fixed-base arithmetic for the provers' secret scalars (64 instead of 11 additions per base).
    pub fn set_constant_time_provers(&self, constant_time: bool) -> Result<(), EngineError> {
        self.check(unsafe { sys::eg_ctx_set_prover_mode(self.ctx, constant_time as i32) })
    }

    /// Tuning knobs (results never depend on them): the ring-proof engine (0 = chosen per chunk, 1 = one launch per equation
    /// index, 2 = one thread per ring, 3 = two lanes per ring) and the number of tallies per call from which
    /// `verify_shares` / `verify_decryptions` build fixed-base tables for the keys (default 32 768, 0 = always).
    pub fn set_ring_engine(&self, mode: i32) -> Result<(), EngineError> {
        self.check(unsafe { sys::eg_ctx_set_ring_mode(self.ctx, mode) })
    }
    pub fn set_key_table_min(&self, min_tallies: usize) -> Result<(), EngineError> {
        self.check(unsafe { sys::eg_ctx_set_key_table_min(self.ctx, min_tallies) })
    }

    fn tally(&self, bytes: &[u8]) -> Vec<Ciphertext<Ristretto>> {
        ciphertexts(bytes)
    }

    // ------------------------------------------------------------------ verification

    /// `cts.iter().zip(proofs).map(|(ct, p)| key.verify_bool(*ct, p))` (keys/impls.rs:101-113).
    pub fn verify_bools(&self, cts: &[Ciphertext<Ristretto>], proofs: &[RingProof<Ristretto>]) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        assert_eq!(cts.len(), proofs.len());
        let n = cts.len();
        let (mut c, mut p) = (Vec::with_capacity(n * 64), Vec::with_capacity(n * 96));
        let mut wrong_len = vec![None; n];
        for (i, (ct, proof)) in cts.iter().zip(proofs).enumerate() {
            c.extend_from_slice(&ct.to_bytes());
            let bytes = proof.to_bytes();
            if bytes.len() != 96 {
                wrong_len[i] = Some(bytes.len() / 32 - 1);      // check_lengths("items in all rings", ..), ring.rs:310-315
                p.resize(p.len() + 96, 0);
            } else {
                p.extend_from_slice(&bytes);
            }
        }
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe { sys::eg_verify_bool_batch(self.ctx, n, c.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts
            .iter()
            .zip(wrong_len)
            .map(|(&v, wrong)| match wrong {
                Some(actual) => Err(VerificationError::LenMismatch { collection: "items in all rings", expected: actual, actual: 2 }),
                None => proof_verdict(v),
            })
            .collect())
    }

    /// `key.verify_zero(ct, proof)` over a batch (keys/impls.rs:59-69).
    pub fn verify_zeros(&self, cts: &[Ciphertext<Ristretto>], proofs: &[LogEqualityProof<Ristretto>]) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        assert_eq!(cts.len(), proofs.len());
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let p: Vec<u8> = proofs.iter().flat_map(|p| p.to_bytes()).collect();
        let mut verdicts = vec![0_u8; cts.len()];
        self.check(unsafe { sys::eg_verify_zero_batch(self.ctx, cts.len(), c.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts.into_iter().map(proof_verdict).collect())
    }

    fn verify_choices_raw<S: elastic_elgamal::app::ProveSum<Ristretto>>(
        &self,
        m: usize,
        single: bool,
        ballots: &[EncryptedChoice<Ristretto, S>],
        sum_bytes: impl Fn(&EncryptedChoice<Ristretto, S>, &mut Vec<u8>),
    ) -> Result<ChoiceOutcome, EngineError> {
        let n = ballots.len();
        let (mut choices, mut rings, mut sums) =
            (Vec::with_capacity(n * m * 64), Vec::with_capacity(n * (1 + 2 * m) * 32), Vec::with_capacity(n * 64));
        let mut wrong_len = vec![false; n];
        for (i, ballot) in ballots.iter().enumerate() {
            let ring = ballot.range_proof().to_bytes();
            if ballot.len() != m || ring.len() != (1 + 2 * m) * 32 {
                // OptionsLenMismatch / LenMismatch are decided on the host (choice.rs:149-158); the slot gets a dummy
                wrong_len[i] = true;
                choices.resize(choices.len() + m * 64, 0);
                rings.resize(rings.len() + (1 + 2 * m) * 32, 0);
                sums.resize(sums.len() + 64, 0);
                continue;
            }
            for ct in ballot.choices_unchecked() {
                choices.extend_from_slice(&ct.to_bytes());
            }
            rings.extend_from_slice(&ring);
            if single {
                sum_bytes(ballot, &mut sums);
            }
        }
        let mut verdicts = vec![0_u8; n];
        let mut tally = vec![0_u8; m * 64];
        self.check(unsafe {
            sys::eg_verify_choice_batch(self.ctx, n, m as u32, single as i32, choices.as_ptr(), rings.as_ptr(),
                                        if single { sums.as_ptr() } else { ptr::null() }, verdicts.as_mut_ptr(), tally.as_mut_ptr())
        })?;
        // a dummy slot is all zeros: it fails verification and therefore never reaches the tally
        let verdicts = verdicts
            .iter()
            .zip(&wrong_len)
            .zip(ballots)
            .map(|((&v, &wrong), ballot)| match (wrong, v) {
                (true, _) => Err(ChoiceVerificationError::OptionsLenMismatch { expected: m, actual: ballot.len() }),
                (_, sys::EG_V_OK) => Ok(()),
                (_, sys::EG_V_CHOICE_SUM) => Err(ChoiceVerificationError::Sum(VerificationError::ChallengeMismatch)),
                _ => Err(ChoiceVerificationError::Range(VerificationError::ChallengeMismatch)),
            })
            .collect();
        Ok(ChoiceOutcome { verdicts, tally: self.tally(&tally) })
    }

    /// `ballots.iter().map(|b| b.verify(params))` + the tally fold, single-choice polling (choice.rs:358-380).
    pub fn verify_choices(
        &self,
        params: &ChoiceParams<Ristretto, SingleChoice>,
        ballots: &[EncryptedChoice<Ristretto, SingleChoice>],
    ) -> Result<ChoiceOutcome, EngineError> {
        self.verify_choices_raw(params.options_count(), true, ballots, |b, out| out.extend_from_slice(&b.sum_proof().to_bytes()))
    }

    /// The same for multi-choice polling (no sum proof).
    pub fn verify_multi_choices(
        &self,
        params: &ChoiceParams<Ristretto, MultiChoice>,
        ballots: &[EncryptedChoice<Ristretto, MultiChoice>],
    ) -> Result<ChoiceOutcome, EngineError> {
        self.verify_choices_raw(params.options_count(), false, ballots, |_, _| {})
    }

    /// `key.verify_range(&range, ct, proof)` over a batch (keys/impls.rs:143-151 -> range.rs:547-577).
    pub fn verify_ranges(
        &self,
        decomposition: &RangeDecomposition,
        transcript_label: &str,
        cts: &[Ciphertext<Ristretto>],
        proofs: &[RangeProof<Ristretto>],
    ) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        assert_eq!(cts.len(), proofs.len());
        let spec = range_spec(decomposition)?;
        let rings = spec.n_rings as usize;
        let total: usize = spec.size[..rings].iter().map(|&s| s as usize).sum();
        let (partial_len, ring_len) = ((rings - 1) * 64, (1 + total) * 32);
        let n = cts.len();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let (mut partials, mut ring_proofs) = (Vec::with_capacity(n * partial_len), Vec::with_capacity(n * ring_len));
        let mut wrong_len = vec![false; n];
        let mut scratch = Vec::new();
        for (i, proof) in proofs.iter().enumerate() {
            scratch.clear();
            flat::to_flat(proof, &mut scratch)?;        // partial ciphertexts | common challenge | ring responses
            if scratch.len() != partial_len + ring_len {
                wrong_len[i] = true;                     // check_lengths("ciphertexts", ..), range.rs:553-558
                scratch.clear();
                scratch.resize(partial_len + ring_len, 0);
            }
            partials.extend_from_slice(&scratch[..partial_len]);
            ring_proofs.extend_from_slice(&scratch[partial_len..]);
        }
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe {
            sys::eg_verify_range_batch(self.ctx, &spec, label.as_ptr(), n, c.as_ptr(), if rings > 1 { partials.as_ptr() } else { ptr::null() },
                                       ring_proofs.as_ptr(), verdicts.as_mut_ptr())
        })?;
        Ok(verdicts
            .iter()
            .zip(wrong_len)
            .map(|(&v, wrong)| if wrong { Err(VerificationError::LenMismatch { collection: "ciphertexts", expected: rings, actual: 0 }) } else { proof_verdict(v) })
            .collect())
    }

    /// `ballots.iter().map(|b| b.verify(params))` + the tally fold (quadratic_voting.rs:291-329).
    pub fn verify_qv_ballots(
        &self,
        params: &QuadraticVotingParams<Ristretto>,
        ballots: &[QuadraticVotingBallot<Ristretto>],
    ) -> Result<QvOutcome, EngineError> {
        let m = params.options_count();
        let mut spec = std::mem::MaybeUninit::<sys::eg_qv_params>::uninit();
        self.check(unsafe { sys::eg_qv_params_new(m as u32, params.credits(), spec.as_mut_ptr()) })?;
        let spec = unsafe { spec.assume_init() };
        let size = unsafe { sys::eg_qv_ballot_size(&spec) };
        let n = ballots.len();
        let mut bytes = Vec::with_capacity(n * size);
        let mut wrong_len = vec![None; n];
        let mut scratch = Vec::new();
        for (i, ballot) in ballots.iter().enumerate() {
            scratch.clear();
            flat::to_flat(ballot, &mut scratch)?;       // votes (ct | range proof)* | credit (ct | range proof) | sum-of-squares proof
            if scratch.len() != size {
                // another number of options (OptionsLenMismatch, quadratic_voting.rs:292-298) or a proof of another shape
                wrong_len[i] = Some(scratch.len());
                scratch.clear();
                scratch.resize(size, 0);
            }
            bytes.extend_from_slice(&scratch);
        }
        let mut verdicts = vec![0_u8; n];
        let mut tally = vec![0_u8; m * 64];
        self.check(unsafe { sys::eg_verify_qv_batch(self.ctx, &spec, n, bytes.as_ptr(), verdicts.as_mut_ptr(), tally.as_mut_ptr()) })?;
        let verdicts = verdicts
            .iter()
            .zip(wrong_len)
            .map(|(&v, wrong)| match (wrong, v) {
                (Some(_), _) => Err(QuadraticVotingError::OptionsLenMismatch { expected: m, actual: usize::MAX }),
                (None, sys::EG_V_OK) => Ok(()),
                (None, sys::EG_V_QV_CREDIT_RANGE) => Err(QuadraticVotingError::CreditRange(VerificationError::ChallengeMismatch)),
                (None, sys::EG_V_QV_CREDIT_EQUIV) => Err(QuadraticVotingError::CreditEquivalence(VerificationError::ChallengeMismatch)),
                (None, v) if v >= sys::EG_V_QV_VARIANT_BASE => {
                    Err(QuadraticVotingError::Variant { index: (v - sys::EG_V_QV_VARIANT_BASE) as usize, error: VerificationError::ChallengeMismatch })
                }
                // a malformed encoding cannot come out of a typed ballot; report it where the reference would fail first
                (None, _) => Err(QuadraticVotingError::Variant { index: 0, error: VerificationError::ChallengeMismatch }),
            })
            .collect();
        Ok(QvOutcome { verdicts, tally: self.tally(&tally) })
    }

    /// `proof.verify(cts.iter(), sum_ct, receiver, &mut Transcript::new(label))` over a batch (mul.rs:190-260).
    pub fn verify_sums_of_squares(
        &self,
        transcript_label: &str,
        count: usize,
        cts: &[Ciphertext<Ristretto>],
        sum_cts: &[Ciphertext<Ristretto>],
        proofs: &[SumOfSquaresProof<Ristretto>],
    ) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        let n = proofs.len();
        assert!(cts.len() == n * count && sum_cts.len() == n);
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let s: Vec<u8> = sum_cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let stride = 32 * (2 * count + 2);
        let mut p = Vec::with_capacity(n * stride);
        let mut wrong_len = vec![None; n];
        let mut scratch = Vec::new();
        for (i, proof) in proofs.iter().enumerate() {
            scratch.clear();
            flat::to_flat(proof, &mut scratch)?;        // challenge | ciphertext responses | sum response
            if scratch.len() != stride {
                wrong_len[i] = Some(scratch.len() / 32 - 2);
                scratch.clear();
                scratch.resize(stride, 0);
            }
            p.extend_from_slice(&scratch);
        }
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe { sys::eg_verify_sumsq_batch(self.ctx, label.as_ptr(), count as u32, n, c.as_ptr(), s.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts
            .iter()
            .zip(wrong_len)
            .map(|(&v, wrong)| match wrong {
                Some(actual) => Err(VerificationError::LenMismatch { collection: "ciphertext responses", expected: 2 * count, actual }),
                None => proof_verdict(v),
            })
            .collect())
    }

    /// `proof.verify(ct, receiver, commitment, blinding_base, &mut Transcript::new(label))` over a batch (commitment.rs:186-238).
    pub fn verify_commitment_equivalences(
        &self,
        transcript_label: &str,
        cts: &[Ciphertext<Ristretto>],
        commitments: &[Element],
        proofs: &[CommitmentEquivalenceProof<Ristretto>],
    ) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        let n = cts.len();
        assert!(commitments.len() == n && proofs.len() == n);
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let mut m = vec![0_u8; n * 32];
        for (chunk, commitment) in m.chunks_mut(32).zip(commitments) {
            Ristretto::serialize_element(commitment, chunk);
        }
        let mut p = Vec::with_capacity(n * 128);
        for proof in proofs {
            flat::to_flat(proof, &mut p)?;              // challenge | randomness, value, commitment responses
        }
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe { sys::eg_verify_commitment_equiv_batch(self.ctx, label.as_ptr(), n, c.as_ptr(), m.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts.into_iter().map(proof_verdict).collect())
    }

    /// `proof.verify(keys.iter(), &mut Transcript::new(label))` over a batch of proofs for `keys_per_proof` keys each
    /// (possession.rs:135-163).
    pub fn verify_possessions(
        &self,
        transcript_label: &str,
        keys_per_proof: usize,
        keys: &[PublicKey<Ristretto>],
        proofs: &[ProofOfPossession<Ristretto>],
    ) -> Result<Vec<Result<(), VerificationError>>, EngineError> {
        let n = proofs.len();
        assert_eq!(keys.len(), n * keys_per_proof);
        let k: Vec<u8> = keys.iter().flat_map(|key| key.as_bytes().iter().copied()).collect();
        let stride = 32 * (1 + keys_per_proof);
        let mut p = Vec::with_capacity(n * stride);
        let mut wrong_len = vec![None; n];
        let mut scratch = Vec::new();
        for (i, proof) in proofs.iter().enumerate() {
            scratch.clear();
            flat::to_flat(proof, &mut scratch)?;        // challenge | responses
            if scratch.len() != stride {
                wrong_len[i] = Some(scratch.len() / 32 - 1);
                scratch.clear();
                scratch.resize(stride, 0);
            }
            p.extend_from_slice(&scratch);
        }
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe { sys::eg_verify_possession_batch(self.ctx, label.as_ptr(), keys_per_proof as u32, n, k.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts
            .iter()
            .zip(wrong_len)
            .map(|(&v, wrong)| match wrong {
                Some(actual) => Err(VerificationError::LenMismatch { collection: "public keys", expected: actual, actual: keys_per_proof }),
                None => proof_verdict(v),
            })
            .collect())
    }

    /// `PublicKeySet::from_participants(params, keys)` over a batch of key sets of one shape (key_set.rs:87-144):
    /// `Ok(shared key)` or `Error::MalformedParticipantKeys`.
    pub fn validate_key_sets(
        &self,
        params: sharing::Params,
        keys: &[PublicKey<Ristretto>],
    ) -> Result<Vec<Result<PublicKey<Ristretto>, sharing::Error>>, EngineError> {
        assert_eq!(keys.len() % params.shares, 0);
        let n = keys.len() / params.shares;
        let k: Vec<u8> = keys.iter().flat_map(|key| key.as_bytes().iter().copied()).collect();
        let mut shared = vec![0_u8; n * 32];
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe {
            sys::eg_keysets_validate_batch(self.ctx, params.shares as u32, params.threshold as u32, n, k.as_ptr(), shared.as_mut_ptr(), verdicts.as_mut_ptr())
        })?;
        Ok(verdicts
            .iter()
            .zip(shared.chunks(32))
            .map(|(&v, key)| if v == sys::EG_V_OK { Ok(PublicKey::from_bytes(key).expect("a reconstructed key is valid")) } else { Err(sharing::Error::MalformedParticipantKeys) })
            .collect())
    }

    fn keyset(key_set: &PublicKeySet<Ristretto>) -> sys::eg_keyset {
        let params = key_set.params();
        let mut ks = sys::eg_keyset { shares: params.shares as u32, threshold: params.threshold as u32, shared_key: [0; 32], participant_keys: [[0; 32]; 64] };
        ks.shared_key.copy_from_slice(key_set.shared_key().as_bytes());
        for (slot, key) in ks.participant_keys.iter_mut().zip(key_set.participant_keys()) {
            slot.copy_from_slice(key.as_bytes());
        }
        ks
    }

    /// `key_set.verify_share(share, ct, index, proof)` for every tally and every listed participant
    /// (key_set.rs:209-228); `shares` / `proofs` are tally-major, `indexes.len()` per tally (at most 8 per call).
    pub fn verify_shares(
        &self,
        key_set: &PublicKeySet<Ristretto>,
        indexes: &[usize],
        cts: &[Ciphertext<Ristretto>],
        shares: &[CandidateDecryption<Ristretto>],
        proofs: &[LogEqualityProof<Ristretto>],
    ) -> Result<Vec<Result<VerifiableDecryption<Ristretto>, VerificationError>>, EngineError> {
        let (n, s) = (cts.len(), indexes.len());
        assert!(key_set.params().shares <= 64 && shares.len() == n * s && proofs.len() == n * s);
        let ks = Self::keyset(key_set);
        let idx: Vec<u32> = indexes.iter().map(|&i| i as u32).collect();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let sh: Vec<u8> = shares.iter().flat_map(|share| share.into_unchecked().to_bytes()).collect();
        let p: Vec<u8> = proofs.iter().flat_map(|p| p.to_bytes()).collect();
        let mut verdicts = vec![0_u8; n * s];
        self.check(unsafe { sys::eg_verify_shares_batch(self.ctx, &ks, n, s as u32, idx.as_ptr(), c.as_ptr(), sh.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr()) })?;
        Ok(verdicts.iter().zip(shares).map(|(&v, share)| proof_verdict(v).map(|()| share.into_unchecked())).collect())
    }

    /// `candidate.verify(ct, key, proof, &mut Transcript::new(label))` over a batch, one custom key (decryption.rs:189-205).
    pub fn verify_decryptions(
        &self,
        transcript_label: &str,
        key: &PublicKey<Ristretto>,
        cts: &[Ciphertext<Ristretto>],
        candidates: &[CandidateDecryption<Ristretto>],
        proofs: &[LogEqualityProof<Ristretto>],
    ) -> Result<Vec<Result<VerifiableDecryption<Ristretto>, VerificationError>>, EngineError> {
        let n = cts.len();
        assert!(candidates.len() == n && proofs.len() == n);
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let d: Vec<u8> = candidates.iter().flat_map(|x| x.into_unchecked().to_bytes()).collect();
        let p: Vec<u8> = proofs.iter().flat_map(|p| p.to_bytes()).collect();
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let mut verdicts = vec![0_u8; n];
        self.check(unsafe {
            sys::eg_verify_decryption_batch(self.ctx, label.as_ptr(), key.as_bytes().as_ptr(), n, c.as_ptr(), d.as_ptr(), p.as_ptr(), verdicts.as_mut_ptr())
        })?;
        Ok(verdicts.iter().zip(candidates).map(|(&v, x)| proof_verdict(v).map(|()| x.into_unchecked())).collect())
    }

    /// `DiscreteLogTable::new(lo..hi)` on the device(s).
    pub fn dlog_table(&self, lo: u64, hi: u64) -> Result<DlogTable<'_>, EngineError> {
        let mut table = ptr::null_mut();
        self.check(unsafe { sys::eg_dlog_table_create(self.ctx, lo, hi, &mut table) })?;
        Ok(DlogTable { engine: self, table })
    }

    /// `DiscreteLogTable::new(lo..hi)` for ranges too large to tabulate: a table of `baby_steps` values and up to
    /// `ceil((hi - lo) / baby_steps)` (<= 2^32) giant steps per lookup; the same answers as a table of every value.
    pub fn dlog_table_bsgs(&self, lo: u64, hi: u64, baby_steps: u64) -> Result<DlogTable<'_>, EngineError> {
        let mut table = ptr::null_mut();
        self.check(unsafe { sys::eg_dlog_table_create_bsgs(self.ctx, lo, hi, baby_steps, &mut table) })?;
        Ok(DlogTable { engine: self, table })
    }

    /// `params.combine_shares(..)` on the listed participants' shares, then `decrypt(ct, &table)` (sharing/mod.rs:302-325,
    /// decryption.rs:138-144), per tally: `Some(value)` or `None` when the plaintext is outside the table.
    pub fn combine_and_decrypt(
        &self,
        indexes: &[usize],
        cts: &[Ciphertext<Ristretto>],
        shares: &[VerifiableDecryption<Ristretto>],
        table: &DlogTable<'_>,
    ) -> Result<Vec<Option<u64>>, EngineError> {
        let (n, t) = (cts.len(), indexes.len());
        assert_eq!(shares.len(), n * t);
        let idx: Vec<u32> = indexes.iter().map(|&i| i as u32).collect();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let sh: Vec<u8> = shares.iter().flat_map(|share| share.to_bytes()).collect();
        let (mut values, mut found) = (vec![0_u64; n], vec![0_u8; n]);
        self.check(unsafe {
            sys::eg_combine_decrypt_batch(self.ctx, t as u32, idx.as_ptr(), n, t as u32, c.as_ptr(), sh.as_ptr(), table.table, values.as_mut_ptr(), found.as_mut_ptr())
        })?;
        Ok(values.iter().zip(found).map(|(&v, f)| (f == 1).then_some(v)).collect())
    }

    /// The tallier of examples/voting.rs: `params.combine_shares(..)` on the shares that `verify_shares` accepted, then
    /// `decrypt(ct, &table)`, per tally.  `shares` is `verify_shares`' output (tally-major, `indexes.len()` per tally, at
    /// most 64); each tally combines its first `threshold` accepted shares in that order.  `Ok(Some(value))`, `Ok(None)` when
    /// the plaintext is outside the table, `Err(CombineError::NotEnoughShares)` when fewer than `threshold` shares were
    /// accepted (`combine_shares` returns `None`).
    pub fn combine_accepted_and_decrypt(
        &self,
        threshold: usize,
        indexes: &[usize],
        cts: &[Ciphertext<Ristretto>],
        shares: &[Result<VerifiableDecryption<Ristretto>, VerificationError>],
        table: &DlogTable<'_>,
    ) -> Result<Vec<Result<Option<u64>, CombineError>>, EngineError> {
        let (n, s) = (cts.len(), indexes.len());
        assert_eq!(shares.len(), n * s);
        let idx: Vec<u32> = indexes.iter().map(|&i| i as u32).collect();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let sh: Vec<u8> = shares.iter().flat_map(|share| share.as_ref().map_or_else(|_| vec![0_u8; 32], |d| d.to_bytes().to_vec())).collect();
        let verdicts: Vec<u8> = shares.iter().map(|share| if share.is_ok() { sys::EG_V_OK } else { sys::EG_V_CHALLENGE_MISMATCH }).collect();
        let (mut values, mut found) = (vec![0_u64; n], vec![0_u8; n]);
        self.check(unsafe {
            sys::eg_combine_decrypt_accepted_batch(self.ctx, threshold as u32, s as u32, idx.as_ptr(), n, c.as_ptr(), sh.as_ptr(), verdicts.as_ptr(),
                                                   table.table, values.as_mut_ptr(), found.as_mut_ptr())
        })?;
        Ok(values
            .iter()
            .zip(found)
            .map(|(&v, f)| {
                debug_assert!(f != 2, "typed ciphertexts and shares decode");
                if f == 3 { Err(CombineError::NotEnoughShares) } else { Ok((f == 1).then_some(v)) }
            })
            .collect())
    }

    // ------------------------------------------------------------------ decryption side (the holder's secret key)

    fn secret_bytes(secret: &SecretKey<Ristretto>) -> [u8; 32] {
        let mut b = [0_u8; 32];
        Ristretto::serialize_scalar(secret.expose_scalar(), &mut b);
        b
    }

    fn share_outputs(dh: &[u8], proofs: &[u8], ok: &[u8]) -> Vec<(VerifiableDecryption<Ristretto>, LogEqualityProof<Ristretto>)> {
        debug_assert!(ok.iter().all(|&f| f == 1), "typed ciphertexts decode");
        dh.chunks(32)
            .zip(proofs.chunks(64))
            .map(|(d, p)| {
                let d = CandidateDecryption::from_bytes(d).expect("the engine emits canonical encodings").into_unchecked();
                (d, LogEqualityProof::from_bytes(p).expect("the engine emits canonical scalars"))
            })
            .collect()
    }

    /// `secret.decrypt_to_element(ct)` over a batch (keys/impls.rs:160-163).
    pub fn decrypt_to_elements(&self, secret: &SecretKey<Ristretto>, cts: &[Ciphertext<Ristretto>]) -> Result<Vec<Element>, EngineError> {
        let n = cts.len();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let (mut elements, mut found) = (vec![0_u8; n * 32], vec![0_u8; n]);
        let key = Self::secret_bytes(secret);
        self.check(unsafe {
            sys::eg_decrypt_batch(self.ctx, key.as_ptr(), n, c.as_ptr(), ptr::null(), elements.as_mut_ptr(), ptr::null_mut(), found.as_mut_ptr())
        })?;
        Ok(elements.chunks(32).map(element).collect())
    }

    /// `secret.decrypt(ct, &table)` over a batch (keys/impls.rs:165-177): `Some(value)` or `None` outside the table.
    pub fn decrypt(&self, secret: &SecretKey<Ristretto>, cts: &[Ciphertext<Ristretto>], table: &DlogTable<'_>) -> Result<Vec<Option<u64>>, EngineError> {
        let n = cts.len();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let (mut values, mut found) = (vec![0_u64; n], vec![0_u8; n]);
        let key = Self::secret_bytes(secret);
        self.check(unsafe {
            sys::eg_decrypt_batch(self.ctx, key.as_ptr(), n, c.as_ptr(), table.table, ptr::null_mut(), values.as_mut_ptr(), found.as_mut_ptr())
        })?;
        Ok(values.iter().zip(found).map(|(&v, f)| (f == 1).then_some(v)).collect())
    }

    /// `participant.decrypt_share(ct, rng)` over a batch for participant `index` of `key_set` holding `secret_share`
    /// (participant.rs:163-185); one randomness block per ciphertext.  A secret share that does not match
    /// `key_set.participant_keys()[index]` is an `EngineError` (the reference cannot build that participant).
    pub fn decrypt_shares(
        &self,
        key_set: &PublicKeySet<Ristretto>,
        index: usize,
        secret_share: &SecretKey<Ristretto>,
        cts: &[Ciphertext<Ristretto>],
        randomness: Randomness<'_>,
    ) -> Result<Vec<(VerifiableDecryption<Ristretto>, LogEqualityProof<Ristretto>)>, EngineError> {
        let n = cts.len();
        assert!(key_set.params().shares <= 64);
        let ks = Self::keyset(key_set);
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let (mut dh, mut proofs, mut ok) = (vec![0_u8; n * 32], vec![0_u8; n * 64], vec![0_u8; n]);
        let key = Self::secret_bytes(secret_share);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * 64);
                unsafe {
                    sys::eg_decrypt_share_batch(self.ctx, &ks, index as u32, key.as_ptr(), n, c.as_ptr(), wide.as_ptr(), dh.as_mut_ptr(),
                                                proofs.as_mut_ptr(), ok.as_mut_ptr())
                }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_decrypt_share_batch_seeded(self.ctx, &ks, index as u32, key.as_ptr(), n, c.as_ptr(), seed.as_ptr(), counter_base,
                                                   dh.as_mut_ptr(), proofs.as_mut_ptr(), ok.as_mut_ptr())
            },
        })?;
        Ok(Self::share_outputs(&dh, &proofs, &ok))
    }

    /// `VerifiableDecryption::new(ct, &keypair, &mut Transcript::new(label), rng)` over a batch with the key pair
    /// `(secret, [secret]G)` (decryption.rs:89-111); one randomness block per ciphertext.
    pub fn prove_decryptions(
        &self,
        transcript_label: &str,
        secret: &SecretKey<Ristretto>,
        cts: &[Ciphertext<Ristretto>],
        randomness: Randomness<'_>,
    ) -> Result<Vec<(VerifiableDecryption<Ristretto>, LogEqualityProof<Ristretto>)>, EngineError> {
        let n = cts.len();
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let (mut dh, mut proofs, mut ok) = (vec![0_u8; n * 32], vec![0_u8; n * 64], vec![0_u8; n]);
        let key = Self::secret_bytes(secret);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * 64);
                unsafe {
                    sys::eg_prove_decryption_batch(self.ctx, label.as_ptr(), key.as_ptr(), n, c.as_ptr(), wide.as_ptr(), dh.as_mut_ptr(),
                                                   proofs.as_mut_ptr(), ok.as_mut_ptr())
                }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_prove_decryption_batch_seeded(self.ctx, label.as_ptr(), key.as_ptr(), n, c.as_ptr(), seed.as_ptr(), counter_base,
                                                      dh.as_mut_ptr(), proofs.as_mut_ptr(), ok.as_mut_ptr())
            },
        })?;
        Ok(Self::share_outputs(&dh, &proofs, &ok))
    }

    // ------------------------------------------------------------------ ciphertext operators

    /// `Σ_j ciphertexts[i][j] * scalars[i][j]` for every row `i` (rows of equal length ≤ 16): the `Add`, `Sub`, `Neg` and
    /// `Mul<&Scalar>` impls of `Ciphertext` (encryption.rs:160-226) over a batch — `a + b` = scalars `(1, 1)`,
    /// `a - b` = `(1, -1)`, `-a` = `(-1)`, `a * k` = `(k)`.
    pub fn combine_ciphertexts(&self, rows: &[(Vec<Scalar>, Vec<Ciphertext<Ristretto>>)]) -> Result<Vec<Ciphertext<Ristretto>>, EngineError> {
        let n = rows.len();
        let terms = rows.first().map_or(1, |r| r.0.len());
        let (mut s, mut c) = (Vec::with_capacity(n * terms * 32), Vec::with_capacity(n * terms * 64));
        for (scalars, cts) in rows {
            assert!(scalars.len() == terms && cts.len() == terms, "rows must have the same number of terms");
            for k in scalars {
                let mut b = [0_u8; 32];
                Ristretto::serialize_scalar(k, &mut b);
                s.extend_from_slice(&b);
            }
            for ct in cts {
                c.extend_from_slice(&ct.to_bytes());
            }
        }
        let (mut out, mut ok) = (vec![0_u8; n * 64], vec![0_u8; n]);
        self.check(unsafe { sys::eg_ciphertexts_lincomb_batch(self.ctx, n, terms as u32, s.as_ptr(), c.as_ptr(), out.as_mut_ptr(), ok.as_mut_ptr()) })?;
        debug_assert!(ok.iter().all(|&f| f == 1), "typed inputs are canonical");
        Ok(ciphertexts(&out))
    }

    /// The weighted tally fold `total[j] += items[i][j] * scalars[i]` (encryption.rs:163,197) over the items whose verdict is
    /// 0 (every item with `None`), e.g. the verdicts of `verify_choices`.  Every item has the same number of ciphertexts
    /// (1..=64).  Variable-time in the scalars: weights are public.
    pub fn weighted_sum(&self, items: &[Vec<Ciphertext<Ristretto>>], scalars: &[Scalar], verdicts: Option<&[u8]>) -> Result<Vec<Ciphertext<Ristretto>>, EngineError> {
        let n = items.len();
        assert!(scalars.len() == n && verdicts.map_or(true, |v| v.len() == n), "one scalar and verdict per item");
        let n_cts = items.first().map_or(1, |r| r.len());
        let (mut s, mut c) = (Vec::with_capacity(n * 32), Vec::with_capacity(n * n_cts * 64));
        for (row, k) in items.iter().zip(scalars) {
            assert!(row.len() == n_cts, "items must have the same number of ciphertexts");
            let mut b = [0_u8; 32];
            Ristretto::serialize_scalar(k, &mut b);
            s.extend_from_slice(&b);
            for ct in row {
                c.extend_from_slice(&ct.to_bytes());
            }
        }
        let (mut out, mut ok) = (vec![0_u8; n_cts * 64], [0_u8; 1]);
        let v = verdicts.map_or(std::ptr::null(), |v| v.as_ptr());
        self.check(unsafe {
            sys::eg_ciphertexts_weighted_sum(self.ctx, n, n_cts as u32, 64 * n_cts, 64, c.as_ptr(), s.as_ptr(), v, out.as_mut_ptr(), ok.as_mut_ptr())
        })?;
        debug_assert!(ok[0] == 1, "typed inputs are canonical");
        Ok(ciphertexts(&out))
    }

    /// The tally fold per group (encryption.rs:163): `totals[g][j]` is the sum of `items[i][j]` over the items with
    /// `groups[i] == g` whose verdict is 0 (every item with `None`), e.g. per-precinct tallies under the verdicts of
    /// `verify_choices`.  Groups without included items are `Ciphertext::zero()`.  Every item has the same number of
    /// ciphertexts (1..=64); `n_groups * n_cts <= 2^22`; a group id `>= n_groups` of an included item is an error.
    pub fn group_sum(&self, items: &[Vec<Ciphertext<Ristretto>>], groups: &[u32], n_groups: u32, verdicts: Option<&[u8]>) -> Result<Vec<Vec<Ciphertext<Ristretto>>>, EngineError> {
        let n = items.len();
        assert!(groups.len() == n && verdicts.map_or(true, |v| v.len() == n), "one group id and verdict per item");
        let n_cts = items.first().map_or(1, |r| r.len());
        let mut c = Vec::with_capacity(n * n_cts * 64);
        for row in items {
            assert!(row.len() == n_cts, "items must have the same number of ciphertexts");
            for ct in row {
                c.extend_from_slice(&ct.to_bytes());
            }
        }
        let (mut out, mut ok) = (vec![0_u8; n_groups as usize * n_cts * 64], vec![0_u8; n_groups as usize]);
        let v = verdicts.map_or(std::ptr::null(), |v| v.as_ptr());
        self.check(unsafe {
            sys::eg_ciphertexts_group_sum(self.ctx, n, n_cts as u32, 64 * n_cts, 64, c.as_ptr(), groups.as_ptr(), n_groups, v, out.as_mut_ptr(),
                                          ok.as_mut_ptr())
        })?;
        debug_assert!(ok.iter().all(|&o| o == 1), "typed inputs decode");
        Ok(out.chunks(n_cts * 64).map(ciphertexts).collect())
    }

    // ------------------------------------------------------------------ creation side

    /// `key.encrypt(value, rng)` over a batch (keys/impls.rs:16-23).
    pub fn encrypt(&self, values: &[u64], randomness: Randomness<'_>) -> Result<Vec<Ciphertext<Ristretto>>, EngineError> {
        let n = values.len();
        let mut cts = vec![0_u8; n * 64];
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * 64);
                unsafe { sys::eg_encrypt_batch(self.ctx, n, values.as_ptr(), wide.as_ptr(), cts.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_encrypt_batch_seeded(self.ctx, n, values.as_ptr(), seed.as_ptr(), counter_base, cts.as_mut_ptr())
            },
        })?;
        Ok(ciphertexts(&cts))
    }

    /// `key.encrypt_bool(value, rng)` over a batch (keys/impls.rs:77-89).
    pub fn encrypt_bools(&self, values: &[bool], randomness: Randomness<'_>) -> Result<Vec<(Ciphertext<Ristretto>, RingProof<Ristretto>)>, EngineError> {
        let n = values.len();
        let v: Vec<u8> = values.iter().map(|&b| b as u8).collect();
        let (mut cts, mut proofs) = (vec![0_u8; n * 64], vec![0_u8; n * 96]);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * 3 * 64);
                unsafe { sys::eg_encrypt_bool_batch(self.ctx, n, v.as_ptr(), wide.as_ptr(), cts.as_mut_ptr(), proofs.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_encrypt_bool_batch_seeded(self.ctx, n, v.as_ptr(), seed.as_ptr(), counter_base, cts.as_mut_ptr(), proofs.as_mut_ptr())
            },
        })?;
        Ok(ciphertexts(&cts).into_iter().zip(proofs.chunks(96).map(|p| RingProof::from_bytes(p).expect("canonical scalars"))).collect())
    }

    /// `EncryptedChoice::single(params, choice, rng)` over a batch (choice.rs:288-306).
    pub fn encrypt_single_choices(
        &self,
        params: &ChoiceParams<Ristretto, SingleChoice>,
        choices: &[usize],
        randomness: Randomness<'_>,
    ) -> Result<Vec<EncryptedChoice<Ristretto, SingleChoice>>, EngineError> {
        let (n, m) = (choices.len(), params.options_count());
        let mut values = vec![0_u8; n * m];
        for (row, &choice) in values.chunks_mut(m).zip(choices) {
            assert!(choice < m, "invalid choice {choice}; expected a value in 0..{m}");      // choice.rs:293-297
            row[choice] = 1;
        }
        let ring_len = 32 * (1 + 2 * m);
        let (mut cts, mut rings, mut sums) = (vec![0_u8; n * m * 64], vec![0_u8; n * ring_len], vec![0_u8; n * 64]);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * (3 * m + 1) * 64);
                unsafe { sys::eg_encrypt_choice_batch(self.ctx, n, m as u32, 1, values.as_ptr(), wide.as_ptr(), cts.as_mut_ptr(), rings.as_mut_ptr(), sums.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_encrypt_choice_batch_seeded(self.ctx, n, m as u32, 1, values.as_ptr(), seed.as_ptr(), counter_base, cts.as_mut_ptr(), rings.as_mut_ptr(), sums.as_mut_ptr())
            },
        })?;
        // EncryptedChoice { choices, range_proof: { common_challenge, ring_responses }, sum_proof: { challenge, response } }
        let mut ballot = Vec::with_capacity(m * 64 + ring_len + 64);
        (0..n)
            .map(|i| {
                ballot.clear();
                ballot.extend_from_slice(&cts[i * m * 64..(i + 1) * m * 64]);
                ballot.extend_from_slice(&rings[i * ring_len..(i + 1) * ring_len]);
                ballot.extend_from_slice(&sums[i * 64..(i + 1) * 64]);
                Ok(flat::from_flat(&ballot, &[m, 2 * m])?)
            })
            .collect()
    }

    /// `key.encrypt_range(&range, value, rng)` over a batch (keys/impls.rs:121-141 = RangeProof::new range.rs:462-473).
    pub fn encrypt_ranges(
        &self,
        decomposition: &RangeDecomposition,
        transcript_label: &str,
        values: &[u64],
        randomness: Randomness<'_>,
    ) -> Result<Vec<(Ciphertext<Ristretto>, RangeProof<Ristretto>)>, EngineError> {
        let spec = range_spec(decomposition)?;
        let rings = spec.n_rings as usize;
        let total: usize = spec.size[..rings].iter().map(|&s| s as usize).sum();
        let (partial_len, ring_len, n) = ((rings - 1) * 64, (1 + total) * 32, values.len());
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let (mut cts, mut partials, mut ring_proofs) = (vec![0_u8; n * 64], vec![0_u8; (n * partial_len).max(1)], vec![0_u8; n * ring_len]);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * unsafe { sys::eg_range_prover_draws(&spec) } * 64);
                unsafe { sys::eg_encrypt_range_batch(self.ctx, &spec, label.as_ptr(), n, values.as_ptr(), wide.as_ptr(), cts.as_mut_ptr(), partials.as_mut_ptr(), ring_proofs.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_encrypt_range_batch_seeded(self.ctx, &spec, label.as_ptr(), n, values.as_ptr(), seed.as_ptr(), counter_base, cts.as_mut_ptr(), partials.as_mut_ptr(), ring_proofs.as_mut_ptr())
            },
        })?;
        let mut proof = Vec::with_capacity(partial_len + ring_len);
        ciphertexts(&cts)
            .into_iter()
            .enumerate()
            .map(|(i, ct)| {
                proof.clear();
                proof.extend_from_slice(&partials[i * partial_len..(i + 1) * partial_len]);
                proof.extend_from_slice(&ring_proofs[i * ring_len..(i + 1) * ring_len]);
                // RangeProof { partial_ciphertexts: Vec<Ciphertext>, inner: RingProof { common_challenge, ring_responses } }
                Ok((ct, flat::from_flat(&proof, &[rings - 1, total])?))
            })
            .collect()
    }

    /// `QuadraticVotingBallot::new(params, votes, rng)` over a batch (quadratic_voting.rs:234-284); `votes` is ballot-major.
    pub fn encrypt_qv_ballots(
        &self,
        params: &QuadraticVotingParams<Ristretto>,
        votes: &[u64],
        randomness: Randomness<'_>,
    ) -> Result<Vec<QuadraticVotingBallot<Ristretto>>, EngineError> {
        let m = params.options_count();
        assert_eq!(votes.len() % m, 0);
        let n = votes.len() / m;
        let mut spec = std::mem::MaybeUninit::<sys::eg_qv_params>::uninit();
        self.check(unsafe { sys::eg_qv_params_new(m as u32, params.credits(), spec.as_mut_ptr()) })?;
        let spec = unsafe { spec.assume_init() };
        let size = unsafe { sys::eg_qv_ballot_size(&spec) };
        let mut ballots = vec![0_u8; n * size];
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * unsafe { sys::eg_qv_prover_draws(&spec) } * 64);
                unsafe { sys::eg_encrypt_qv_batch(self.ctx, &spec, n, votes.as_ptr(), wide.as_ptr(), ballots.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_encrypt_qv_batch_seeded(self.ctx, &spec, n, votes.as_ptr(), seed.as_ptr(), counter_base, ballots.as_mut_ptr())
            },
        })?;
        // sequence lengths in visiting order: votes; per vote (partial ciphertexts, ring responses); credit (the same two);
        // the sum-of-squares proof's ciphertext responses
        let (vr, cr) = (&spec.vote_range, &spec.credit_range);
        let total = |r: &sys::eg_range| r.size[..r.n_rings as usize].iter().map(|&s| s as usize).sum::<usize>();
        let mut lens = vec![m];
        for _ in 0..m {
            lens.extend([vr.n_rings as usize - 1, total(vr)]);
        }
        lens.extend([cr.n_rings as usize - 1, total(cr), 2 * m]);
        ballots.chunks(size).map(|b| Ok(flat::from_flat(b, &lens)?)).collect()
    }

    // ------------------------------------------------------------------ stand-alone sigma provers

    fn scalar_bytes(secrets: &[SecretKey<Ristretto>]) -> Vec<u8> {
        secrets.iter().flat_map(Self::secret_bytes).collect()
    }

    fn secret_key(bytes: &[u8]) -> SecretKey<Ristretto> {
        SecretKey::new(Ristretto::deserialize_scalar(bytes).expect("the engine emits canonical scalars"))
    }

    /// `CommitmentEquivalenceProof::new(ciphertext_with_value, receiver, blinding_base, &mut Transcript::new(label), rng)`
    /// over a batch (commitment.rs:126-196) for ciphertexts of `values[i]` with randomness `ct_randomness[i]`; four randomness
    /// blocks per item (blinding, e_r, e_v, e_c).  Returns the re-encrypted ciphertext, the proof, the commitment
    /// `[v]G + [b]H` and the blinding `b` (secret).  Needs the receiver key and the blinding base.
    pub fn prove_commitment_equivalences(
        &self,
        transcript_label: &str,
        values: &[u64],
        ct_randomness: &[SecretKey<Ristretto>],
        randomness: Randomness<'_>,
    ) -> Result<Vec<(Ciphertext<Ristretto>, CommitmentEquivalenceProof<Ristretto>, Element, SecretKey<Ristretto>)>, EngineError> {
        let n = values.len();
        assert_eq!(ct_randomness.len(), n);
        let r = Self::scalar_bytes(ct_randomness);
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let (mut cts, mut coms, mut proofs, mut blind) = (vec![0_u8; n * 64], vec![0_u8; n * 32], vec![0_u8; n * 128], vec![0_u8; n * 32]);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * 4 * 64);
                unsafe {
                    sys::eg_prove_commitment_equiv_batch(self.ctx, label.as_ptr(), n, values.as_ptr(), r.as_ptr(), wide.as_ptr(), cts.as_mut_ptr(),
                                                         coms.as_mut_ptr(), proofs.as_mut_ptr(), blind.as_mut_ptr())
                }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_prove_commitment_equiv_batch_seeded(self.ctx, label.as_ptr(), n, values.as_ptr(), r.as_ptr(), seed.as_ptr(), counter_base,
                                                            cts.as_mut_ptr(), coms.as_mut_ptr(), proofs.as_mut_ptr(), blind.as_mut_ptr())
            },
        })?;
        let out = ciphertexts(&cts)
            .into_iter()
            .zip(proofs.chunks(128).zip(coms.chunks(32)).zip(blind.chunks(32)))
            .map(|(ct, ((p, c), b))| Ok((ct, flat::from_flat(p, &[])?, element(c), Self::secret_key(b))))
            .collect();
        blind.iter_mut().for_each(|x| *x = 0);
        out
    }

    /// `SumOfSquaresProof::new(ciphertexts, sum_of_squares, receiver, &mut Transcript::new(label), rng)` over a batch
    /// (mul.rs:107-181): item `i` has the `count` ciphertexts `cts[i * count..]` of `values` with `ct_randomness`, and the sum
    /// ciphertext `sum_cts[i]` with `sum_randomness[i]`; `1 + 2 count` randomness blocks per item.  As in the reference, the
    /// inputs are not checked against each other: an inconsistent item yields a proof that does not verify.
    #[allow(clippy::too_many_arguments)]
    pub fn prove_sums_of_squares(
        &self,
        transcript_label: &str,
        count: usize,
        cts: &[Ciphertext<Ristretto>],
        values: &[u64],
        ct_randomness: &[SecretKey<Ristretto>],
        sum_cts: &[Ciphertext<Ristretto>],
        sum_randomness: &[SecretKey<Ristretto>],
        randomness: Randomness<'_>,
    ) -> Result<Vec<SumOfSquaresProof<Ristretto>>, EngineError> {
        let n = sum_cts.len();
        assert!(cts.len() == n * count && values.len() == n * count && ct_randomness.len() == n * count && sum_randomness.len() == n);
        let c: Vec<u8> = cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let s: Vec<u8> = sum_cts.iter().flat_map(|ct| ct.to_bytes()).collect();
        let (r, sr) = (Self::scalar_bytes(ct_randomness), Self::scalar_bytes(sum_randomness));
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let stride = 32 * (2 * count + 2);
        let mut proofs = vec![0_u8; n * stride];
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * (1 + 2 * count) * 64);
                unsafe {
                    sys::eg_prove_sumsq_batch(self.ctx, label.as_ptr(), count as u32, n, c.as_ptr(), values.as_ptr(), r.as_ptr(), s.as_ptr(),
                                              sr.as_ptr(), wide.as_ptr(), proofs.as_mut_ptr())
                }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_prove_sumsq_batch_seeded(self.ctx, label.as_ptr(), count as u32, n, c.as_ptr(), values.as_ptr(), r.as_ptr(), s.as_ptr(),
                                                 sr.as_ptr(), seed.as_ptr(), counter_base, proofs.as_mut_ptr())
            },
        })?;
        // SumOfSquaresProof { challenge, ciphertext_responses: Vec<Scalar>, sum_response }
        proofs.chunks(stride).map(|p| Ok(flat::from_flat(p, &[2 * count])?)).collect()
    }

    /// `Keypair::from(secret)` for each of `keys_per_proof` secrets, then `ProofOfPossession::from_keys(keypairs,
    /// &mut Transcript::new(label), rng)` (possession.rs:93-130), over a batch; one randomness block per key.  The public keys
    /// are computed on the device.
    pub fn prove_possessions(
        &self,
        transcript_label: &str,
        keys_per_proof: usize,
        secrets: &[SecretKey<Ristretto>],
        randomness: Randomness<'_>,
    ) -> Result<Vec<(Vec<PublicKey<Ristretto>>, ProofOfPossession<Ristretto>)>, EngineError> {
        let k = keys_per_proof;
        assert!(k > 0 && secrets.len() % k == 0);
        let n = secrets.len() / k;
        let s = Self::scalar_bytes(secrets);
        let label = CString::new(transcript_label).map_err(|_| EngineError { status: sys::EG_ERR_INVALID_ARG, message: "label contains NUL".into() })?;
        let (mut keys, mut proofs) = (vec![0_u8; n * k * 32], vec![0_u8; n * (1 + k) * 32]);
        self.check(match randomness {
            Randomness::Blocks(wide) => {
                assert_eq!(wide.len(), n * k * 64);
                unsafe { sys::eg_prove_possession_batch(self.ctx, label.as_ptr(), k as u32, n, s.as_ptr(), wide.as_ptr(), keys.as_mut_ptr(), proofs.as_mut_ptr()) }
            }
            Randomness::Seeded { seed, counter_base } => unsafe {
                sys::eg_prove_possession_batch_seeded(self.ctx, label.as_ptr(), k as u32, n, s.as_ptr(), seed.as_ptr(), counter_base,
                                                      keys.as_mut_ptr(), proofs.as_mut_ptr())
            },
        })?;
        keys.chunks(32 * k)
            .zip(proofs.chunks(32 * (1 + k)))
            .zip(secrets.chunks(k))
            .map(|((ks, p), sec)| {
                // a zero secret's key is the identity, which PublicKey::from_bytes refuses: take Keypair::from's key then
                let keys = ks.chunks(32).zip(sec).map(|(b, s)| PublicKey::from_bytes(b).unwrap_or_else(|_| PublicKey::from(s))).collect();
                Ok((keys, flat::from_flat(p, &[k])?))
            })
            .collect()
    }

    /// Raw pass-through for objects a caller already holds in the flat layouts (e.g. straight from storage).
    pub fn raw(&self) -> *mut sys::eg_ctx {
        self.ctx
    }
}

impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { sys::eg_ctx_destroy(self.ctx) }
    }
}

/// Flat form of any serde-serialisable object of the reference (element / scalar fields in struct order).
pub fn flat_bytes<T: Serialize>(value: &T) -> Result<Vec<u8>, flat::FlatError> {
    let mut out = Vec::new();
    flat::to_flat(value, &mut out)?;
    Ok(out)
}
