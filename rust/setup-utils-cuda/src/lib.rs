//! # setup-utils-cuda
//!
//! Safe wrappers over `libsnarksetup_b200.so` with the *reference's own signatures*, so that the bodies of
//! `setup_utils::{generate_powers_of_tau, batch_exp, batch_mul, merge_pairs, power_pairs, check_subgroup, same_ratio,
//! check_same_ratio}` (setup-utils/src/helpers.rs:32,56,75,371,388,406,410; elements.rs:123),
//! `phase1::helpers::buffers::apply_powers` (phase1/src/helpers/buffers.rs:77), `Phase1::computation`
//! (phase1/src/computation.rs:16-25) and the per-vector half of `Phase1::verification`
//! (phase1/src/verification.rs:26-40,217-411) become one call each; further down the SURVEY §8f rows: verdicts from
//! ratio pairs, accumulator re-layout (`Phase1::aggregation` / `split` / `decompress`), `Groth16Params::new`, group
//! IFFT / H query and the QAP row sums of phase 2, and phase 2's `MPCParameters::contribute` / `verify` on the H and L
//! queries (`phase2_contribute`, `phase2_verify`, sharded through `phase2_verification_pairs`).
//!
//! The seam is at byte-slice granularity: arkworks' `Affine<P>` is not `repr(C)`, so the generic in-memory entry
//! points serialise to the canonical uncompressed form, call the engine, and read the result back; the phase1
//! entry points already work on the CLI's byte buffers (mmaps) and pass them straight through.
//!
//! There is no CPU fallback: a device failure (code 9) panics, as a failed `expect` does in the reference's
//! rayon tasks (computation.rs:99,142,161,180).
pub mod ffi;

use ark_ec::{pairing::Pairing, AffineRepr};
use ark_ff::{PrimeField, Zero};
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize, Compress, SerializationError, Validate};
use phase1::{Phase1Parameters, PrivateKey};
use rand::{rngs::OsRng, RngCore};
use setup_utils::{
    converters::{ContributionMode, ProvingSystem},
    BatchExpMode, CheckForCorrectness, Error, Result, SubgroupCheckMode, UseCompression, VerificationError,
};
use std::os::raw::c_int;

// ------------------------------------------------------------------------------------------------------------------
// curve / group ids of the C ABI
// ------------------------------------------------------------------------------------------------------------------

/// Pairing engines the engine implements (ss_curve).
pub trait CudaCurve: Pairing {
    const CURVE_ID: c_int;
}
impl CudaCurve for ark_bls12_377::Bls12_377 {
    const CURVE_ID: c_int = ffi::SS_CURVE_BLS12_377;
}
impl CudaCurve for ark_bw6_761::BW6_761 {
    const CURVE_ID: c_int = ffi::SS_CURVE_BW6_761;
}

/// Affine groups the engine implements (ss_curve, ss_group).
pub trait CudaGroup: AffineRepr {
    const CURVE_ID: c_int;
    const GROUP_ID: c_int;
}
impl CudaGroup for ark_bls12_377::G1Affine {
    const CURVE_ID: c_int = ffi::SS_CURVE_BLS12_377;
    const GROUP_ID: c_int = ffi::SS_G1;
}
impl CudaGroup for ark_bls12_377::G2Affine {
    const CURVE_ID: c_int = ffi::SS_CURVE_BLS12_377;
    const GROUP_ID: c_int = ffi::SS_G2;
}
impl CudaGroup for ark_bw6_761::G1Affine {
    const CURVE_ID: c_int = ffi::SS_CURVE_BW6_761;
    const GROUP_ID: c_int = ffi::SS_G1;
}
impl CudaGroup for ark_bw6_761::G2Affine {
    const CURVE_ID: c_int = ffi::SS_CURVE_BW6_761;
    const GROUP_ID: c_int = ffi::SS_G2;
}

// ------------------------------------------------------------------------------------------------------------------
// helpers
// ------------------------------------------------------------------------------------------------------------------

fn last_error() -> ffi::SsErrorInfo {
    let mut e: ffi::SsErrorInfo = unsafe { std::mem::zeroed() };
    unsafe { ffi::ss_last_error(&mut e) };
    e
}

fn message(e: &ffi::SsErrorInfo) -> String {
    let bytes: Vec<u8> = e.message.iter().take_while(|c| **c != 0).map(|c| *c as u8).collect();
    String::from_utf8_lossy(&bytes).into_owned()
}

/// ss_status -> setup_utils::Error (setup-utils/src/errors.rs:11-38,97-100), 1:1 with include/snark_setup_b200.h.
fn check(rc: c_int) -> Result<()> {
    match rc {
        0 => Ok(()),
        1 => Err(Error::ZexeSerializationError(SerializationError::InvalidData)),
        2 => Err(Error::ZexeSerializationError(SerializationError::UnexpectedFlags)),
        3 => Err(Error::PointAtInfinity),
        4 => Err(Error::IncorrectSubgroup),
        5 => {
            let e = last_error();
            Err(Error::InvalidLength { expected: e.expected as usize, got: e.got as usize })
        }
        6 => Err(Error::InvalidChunk),
        7 => Err(Error::BatchTooSmall),
        10 => Err(VerificationError::InvalidRatio(message(&last_error())).into()),
        _ => panic!("snark-setup CUDA engine failure (code {}): {} — there is no CPU fallback", rc, message(&last_error())),
    }
}

fn flag(c: UseCompression) -> c_int {
    match c {
        Compress::Yes => 1,
        Compress::No => 0,
    }
}

fn check_mode(c: CheckForCorrectness) -> c_int {
    match c {
        CheckForCorrectness::Full => 0,
        CheckForCorrectness::OnlyNonZero => 1,
        CheckForCorrectness::OnlyInGroup => 2,
        CheckForCorrectness::No => 3,
    }
}

fn subgroup_mode(m: SubgroupCheckMode) -> c_int {
    match m {
        SubgroupCheckMode::Auto => 0,
        SubgroupCheckMode::Direct => 1,
        SubgroupCheckMode::Batched => 2,
        SubgroupCheckMode::No => 3,
    }
}

/// canonical little-endian bytes of a scalar (= `Fr::serialize_uncompressed`: 32 B BLS12-377, 48 B BW6-761)
fn scalar_bytes<F: PrimeField>(s: &F) -> Vec<u8> {
    let mut v = Vec::with_capacity(F::zero().uncompressed_size());
    s.serialize_uncompressed(&mut v).expect("scalar serialisation cannot fail");
    v
}

fn scalars_bytes<F: PrimeField>(s: &[F]) -> Vec<u8> {
    let mut v = Vec::with_capacity(s.len() * F::zero().uncompressed_size());
    for x in s {
        x.serialize_uncompressed(&mut v).expect("scalar serialisation cannot fail");
    }
    v
}

fn points_bytes<C: AffineRepr>(p: &[C]) -> Vec<u8> {
    let mut v = Vec::with_capacity(p.len() * C::zero().uncompressed_size());
    for x in p {
        x.serialize_uncompressed(&mut v).expect("point serialisation cannot fail");
    }
    v
}

fn points_from<C: AffineRepr>(bytes: &[u8], out: &mut [C]) -> Result<()> {
    let sz = C::zero().uncompressed_size();
    for (i, o) in out.iter_mut().enumerate() {
        *o = C::deserialize_with_mode(&bytes[i * sz..(i + 1) * sz], Compress::No, Validate::No)?;
    }
    Ok(())
}

fn read_points<C: AffineRepr>(bytes: &[u8], n: usize) -> Vec<C> {
    let mut out = vec![C::zero(); n];
    points_from(bytes, &mut out).expect("engine returns canonical points");
    out
}

fn params_of<E: CudaCurve>(p: &Phase1Parameters<E>) -> ffi::SsPhase1Params {
    ffi::SsPhase1Params {
        curve: E::CURVE_ID,
        proving_system: match p.proving_system {
            ProvingSystem::Groth16 => 0,
            ProvingSystem::Marlin => 1,
        },
        contribution_mode: match p.contribution_mode {
            ContributionMode::Full => 0,
            ContributionMode::Chunked => 1,
        },
        chunk_index: p.chunk_index as u64,
        chunk_size: p.chunk_size as u64,
        total_size_in_log2: p.total_size_in_log2 as u32,
        batch_size: p.batch_size as u64,
    }
}

fn rho_seed() -> [u8; 32] {
    // the reference draws the random linear combination from thread_rng (helpers.rs:373); the engine expands a
    // 32-byte OS-random key with ChaCha20 on the device
    let mut s = [0u8; 32];
    OsRng.fill_bytes(&mut s);
    s
}

/// Select the GPUs of this process (ss_init); without it the engine uses $SNARK_SETUP_GPUS or device 0.
pub fn init(devices: &[i32]) -> Result<()> {
    check(unsafe { ffi::ss_init(devices.as_ptr(), devices.len() as c_int) })
}

/// See include/snark_setup_b200.h: bases read without a subgroup check go through the reference's double-and-add.
pub fn set_strict_unchecked_inputs(on: bool) {
    unsafe { ffi::ss_set_strict_unchecked_inputs(on as c_int) }
}

// ------------------------------------------------------------------------------------------------------------------
// setup-utils helpers (same signatures as setup-utils/src/helpers.rs and elements.rs)
// ------------------------------------------------------------------------------------------------------------------

/// setup_utils::generate_powers_of_tau — helpers.rs:32-37
pub fn generate_powers_of_tau<E: CudaCurve>(tau: &E::ScalarField, start: usize, end: usize) -> Vec<E::ScalarField> {
    let n = end.saturating_sub(start);
    let fb = E::ScalarField::zero().uncompressed_size();
    let mut out = vec![0u8; n * fb];
    let t = scalar_bytes(tau);
    check(unsafe { ffi::ss_generate_powers_of_tau(E::CURVE_ID, t.as_ptr(), start as u64, end as u64, out.as_mut_ptr()) })
        .expect("generate_powers_of_tau");
    (0..n)
        .map(|i| E::ScalarField::deserialize_uncompressed(&out[i * fb..(i + 1) * fb]).expect("canonical scalar"))
        .collect()
}

/// setup_utils::batch_exp — helpers.rs:75-140 (`batch_exp_mode` selects nothing in the reference either, :89-92)
pub fn batch_exp<C: CudaGroup>(
    bases: &mut [C],
    exps: &[C::ScalarField],
    coeff: Option<&C::ScalarField>,
    _batch_exp_mode: BatchExpMode,
) -> Result<()> {
    if bases.len() != exps.len() {
        return Err(Error::InvalidLength { expected: bases.len(), got: exps.len() });
    }
    let mut buf = points_bytes(bases);
    let e = scalars_bytes(exps);
    let c = coeff.map(scalar_bytes);
    check(unsafe {
        ffi::ss_batch_exp(
            C::CURVE_ID,
            C::GROUP_ID,
            buf.as_mut_ptr(),
            bases.len(),
            e.as_ptr(),
            exps.len(),
            c.as_ref().map_or(std::ptr::null(), |v| v.as_ptr()),
        )
    })?;
    points_from(&buf, bases)
}

/// setup_utils::batch_mul — helpers.rs:56-59 (phase2 delta^-1 of the H and L queries, parameters.rs:294-296)
pub fn batch_mul<C: CudaGroup>(bases: &mut [C], coeff: &C::ScalarField, _batch_exp_mode: BatchExpMode) -> Result<()> {
    let mut buf = points_bytes(bases);
    let c = scalar_bytes(coeff);
    check(unsafe { ffi::ss_batch_mul(C::CURVE_ID, C::GROUP_ID, buf.as_mut_ptr(), bases.len(), c.as_ptr()) })?;
    points_from(&buf, bases)
}

/// The streaming form phase2 uses (chunked_groth16.rs:442-466): the query already sits in a byte buffer.
pub fn batch_mul_bytes<C: CudaGroup>(bases_uncompressed: &mut [u8], coeff: &C::ScalarField) -> Result<()> {
    let n = bases_uncompressed.len() / C::zero().uncompressed_size();
    let c = scalar_bytes(coeff);
    check(unsafe { ffi::ss_batch_mul(C::CURVE_ID, C::GROUP_ID, bases_uncompressed.as_mut_ptr(), n, c.as_ptr()) })
}

/// setup_utils::merge_pairs — helpers.rs:371-384
pub fn merge_pairs<G: CudaGroup>(v1: &[G], v2: &[G]) -> (G, G) {
    assert_eq!(v1.len(), v2.len());
    let (a, b) = (points_bytes(v1), points_bytes(v2));
    let usz = G::zero().uncompressed_size();
    let (mut s, mut sx) = (vec![0u8; usz], vec![0u8; usz]);
    let seed = rho_seed();
    check(unsafe {
        ffi::ss_merge_pairs(
            G::CURVE_ID,
            G::GROUP_ID,
            a.as_ptr(),
            b.as_ptr(),
            0,
            check_mode(CheckForCorrectness::No),
            v1.len(),
            std::ptr::null(),
            seed.as_ptr(),
            s.as_mut_ptr(),
            sx.as_mut_ptr(),
        )
    })
    .expect("merge_pairs");
    (
        G::deserialize_with_mode(&s[..], Compress::No, Validate::No).expect("engine returns canonical points"),
        G::deserialize_with_mode(&sx[..], Compress::No, Validate::No).expect("engine returns canonical points"),
    )
}

/// setup_utils::power_pairs — helpers.rs:388-390
pub fn power_pairs<G: CudaGroup>(v: &[G]) -> (G, G) {
    let a = points_bytes(v);
    let usz = G::zero().uncompressed_size();
    let (mut s, mut sx) = (vec![0u8; usz], vec![0u8; usz]);
    let seed = rho_seed();
    check(unsafe {
        ffi::ss_power_pairs(
            G::CURVE_ID,
            G::GROUP_ID,
            a.as_ptr(),
            0,
            check_mode(CheckForCorrectness::No),
            v.len(),
            std::ptr::null(),
            seed.as_ptr(),
            s.as_mut_ptr(),
            sx.as_mut_ptr(),
        )
    })
    .expect("power_pairs");
    (
        G::deserialize_with_mode(&s[..], Compress::No, Validate::No).expect("engine returns canonical points"),
        G::deserialize_with_mode(&sx[..], Compress::No, Validate::No).expect("engine returns canonical points"),
    )
}

/// setup_utils::check_subgroup — elements.rs:123-150
pub fn check_subgroup<C: CudaGroup>(elements: &[C], subgroup_check_mode: SubgroupCheckMode) -> core::result::Result<(), Error> {
    let a = points_bytes(elements);
    check(unsafe {
        ffi::ss_check_subgroup(C::CURVE_ID, C::GROUP_ID, a.as_ptr(), 0, elements.len(), subgroup_mode(subgroup_check_mode))
    })
}

fn pair_bytes<A: AffineRepr>(p: &(A, A)) -> Vec<u8> {
    points_bytes(&[p.0, p.1])
}

/// setup_utils::same_ratio — helpers.rs:406-408
pub fn same_ratio<E: CudaCurve>(g1: &(E::G1Affine, E::G1Affine), g2: &(E::G2Affine, E::G2Affine)) -> bool {
    let (a, b) = (pair_bytes(g1), pair_bytes(g2));
    let mut same: c_int = 0;
    check(unsafe { ffi::ss_same_ratio(E::CURVE_ID, a.as_ptr(), b.as_ptr(), &mut same) }).expect("same_ratio");
    same != 0
}

/// setup_utils::check_same_ratio — helpers.rs:410-424
pub fn check_same_ratio<E: CudaCurve>(
    g1: &(E::G1Affine, E::G1Affine),
    g2: &(E::G2Affine, E::G2Affine),
    err: String,
) -> Result<()> {
    let (a, b) = (pair_bytes(g1), pair_bytes(g2));
    match unsafe { ffi::ss_check_same_ratio(E::CURVE_ID, a.as_ptr(), b.as_ptr()) } {
        10 => Err(VerificationError::InvalidRatio(err).into()),
        rc => check(rc),
    }
}

// ------------------------------------------------------------------------------------------------------------------
// phase1 helpers
// ------------------------------------------------------------------------------------------------------------------

/// phase1::helpers::buffers::apply_powers — buffers.rs:77-97 (same tuple arguments).
pub fn apply_powers<C: CudaGroup>(
    (output, output_compressed): (&mut [u8], UseCompression),
    (input, input_compressed, check_input_for_correctness): (&[u8], UseCompression, CheckForCorrectness),
    (start, end): (usize, usize),
    powers: &[C::ScalarField],
    coeff: Option<&C::ScalarField>,
    _batch_exp_mode: BatchExpMode,
) -> Result<()> {
    let in_size = setup_utils::buffer_size::<C>(input_compressed);
    let out_size = setup_utils::buffer_size::<C>(output_compressed);
    let n = end - start;
    let p = scalars_bytes(&powers[..n]);
    let c = coeff.map(scalar_bytes);
    check(unsafe {
        ffi::ss_apply_powers(
            C::CURVE_ID,
            C::GROUP_ID,
            input[start * in_size..end * in_size].as_ptr(),
            flag(input_compressed),
            check_mode(check_input_for_correctness),
            output[start * out_size..end * out_size].as_mut_ptr(),
            flag(output_compressed),
            n,
            p.as_ptr(),
            std::ptr::null(),
            0,
            c.as_ref().map_or(std::ptr::null(), |v| v.as_ptr()),
        )
    })
}

/// apply_powers with the scalars tau^(start + i) generated on the device (fused generate_powers_of_tau, helpers.rs:32-37):
/// what `Phase1::computation` wants — the powers vector never exists on the host.
pub fn apply_powers_of_tau<C: CudaGroup>(
    (output, output_compressed): (&mut [u8], UseCompression),
    (input, input_compressed, check_input_for_correctness): (&[u8], UseCompression, CheckForCorrectness),
    (start, end): (usize, usize),
    tau: &C::ScalarField,
    first_power: u64,
    coeff: Option<&C::ScalarField>,
) -> Result<()> {
    let in_size = setup_utils::buffer_size::<C>(input_compressed);
    let out_size = setup_utils::buffer_size::<C>(output_compressed);
    let t = scalar_bytes(tau);
    let c = coeff.map(scalar_bytes);
    check(unsafe {
        ffi::ss_apply_powers(
            C::CURVE_ID,
            C::GROUP_ID,
            input[start * in_size..end * in_size].as_ptr(),
            flag(input_compressed),
            check_mode(check_input_for_correctness),
            output[start * out_size..end * out_size].as_mut_ptr(),
            flag(output_compressed),
            end - start,
            std::ptr::null(),
            t.as_ptr(),
            first_power,
            c.as_ref().map_or(std::ptr::null(), |v| v.as_ptr()),
        )
    })
}

/// `Phase1::computation` — phase1/src/computation.rs:16-25, same argument order (BatchExpMode is ignored there too).
#[allow(clippy::too_many_arguments)]
pub fn phase1_computation<E: CudaCurve>(
    input: &[u8],
    output: &mut [u8],
    compressed_input: UseCompression,
    compressed_output: UseCompression,
    check_input_for_correctness: CheckForCorrectness,
    _batch_exp_mode: BatchExpMode,
    key: &PrivateKey<E>,
    parameters: &Phase1Parameters<E>,
) -> Result<()> {
    phase1_computation_shard(
        input,
        output,
        compressed_input,
        compressed_output,
        check_input_for_correctness,
        key,
        parameters,
        (0, 1),
    )
}

/// Index-range shard `shard.0` of `shard.1` of the same computation (one process per GPU, all mapping the same files).
#[allow(clippy::too_many_arguments)]
pub fn phase1_computation_shard<E: CudaCurve>(
    input: &[u8],
    output: &mut [u8],
    compressed_input: UseCompression,
    compressed_output: UseCompression,
    check_input_for_correctness: CheckForCorrectness,
    key: &PrivateKey<E>,
    parameters: &Phase1Parameters<E>,
    shard: (u32, u32),
) -> Result<()> {
    let p = params_of(parameters);
    let (t, a, b) = (scalar_bytes(&key.tau), scalar_bytes(&key.alpha), scalar_bytes(&key.beta));
    check(unsafe {
        ffi::ss_phase1_computation_shard(
            &p,
            input.as_ptr(),
            input.len(),
            output.as_mut_ptr(),
            output.len(),
            flag(compressed_input),
            flag(compressed_output),
            check_mode(check_input_for_correctness),
            t.as_ptr(),
            a.as_ptr(),
            b.as_ptr(),
            shard.0,
            shard.1,
        )
    })
}

/// `Phase1::initialization` — phase1/src/initialization.rs:12-57
pub fn phase1_initialization<E: CudaCurve>(
    output: &mut [u8],
    compressed_output: UseCompression,
    parameters: &Phase1Parameters<E>,
) -> Result<()> {
    let p = params_of(parameters);
    check(unsafe { ffi::ss_phase1_initialization(&p, output.as_mut_ptr(), output.len(), flag(compressed_output)) })
}

/// The `(s, sx)` pairs of the four power vectors of a response: tau_g1, tau_g2, alpha_g1, beta_g1.
pub struct RatioPairs<E: Pairing> {
    pub tau_g1: (E::G1Affine, E::G1Affine),
    pub tau_g2: (E::G2Affine, E::G2Affine),
    pub alpha_g1: (E::G1Affine, E::G1Affine),
    pub beta_g1: (E::G1Affine, E::G1Affine),
}

fn read_pairs<E: CudaCurve>(blob: &[u8]) -> RatioPairs<E> {
    let u1 = E::G1Affine::zero().uncompressed_size();
    let u2 = E::G2Affine::zero().uncompressed_size();
    let g1 = |o: usize| E::G1Affine::deserialize_with_mode(&blob[o..o + u1], Compress::No, Validate::No).expect("canonical point");
    let g2 = |o: usize| E::G2Affine::deserialize_with_mode(&blob[o..o + u2], Compress::No, Validate::No).expect("canonical point");
    RatioPairs {
        tau_g1: (g1(0), g1(u1)),
        tau_g2: (g2(2 * u1), g2(2 * u1 + u2)),
        alpha_g1: (g1(2 * u1 + 2 * u2), g1(3 * u1 + 2 * u2)),
        beta_g1: (g1(4 * u1 + 2 * u2), g1(5 * u1 + 2 * u2)),
    }
}

/// The per-vector loop of `Phase1::verification` (phase1/src/verification.rs:217-411) over the whole response: nonzero
/// and subgroup checks of every element, the vectors re-encoded into `new_challenge`, and ONE `(s, sx)` pair per
/// vector — the caller runs its four `check_same_ratio` on them instead of two pairings per `batch_size` window.
/// The proof-of-knowledge checks on the first elements (verification.rs:83-213) stay where they are.
#[allow(clippy::too_many_arguments)]
pub fn phase1_verification_vectors<E: CudaCurve>(
    output: &[u8],
    new_challenge: Option<&mut [u8]>,
    compressed_output: UseCompression,
    compressed_new_challenge: UseCompression,
    subgroup_check_mode: SubgroupCheckMode,
    ratio_check: bool,
    parameters: &Phase1Parameters<E>,
) -> Result<RatioPairs<E>> {
    let blob = phase1_verification_vectors_shard(
        output,
        new_challenge,
        compressed_output,
        compressed_new_challenge,
        subgroup_check_mode,
        ratio_check,
        parameters,
        (0, 1),
    )?;
    Ok(read_pairs::<E>(&blob))
}

/// Shard `shard.0` of `shard.1`: returns the PARTIAL pairs blob; `reduce_partial_pairs` adds the shards' blobs.
#[allow(clippy::too_many_arguments)]
pub fn phase1_verification_vectors_shard<E: CudaCurve>(
    output: &[u8],
    new_challenge: Option<&mut [u8]>,
    compressed_output: UseCompression,
    compressed_new_challenge: UseCompression,
    subgroup_check_mode: SubgroupCheckMode,
    ratio_check: bool,
    parameters: &Phase1Parameters<E>,
    shard: (u32, u32),
) -> Result<Vec<u8>> {
    let p = params_of(parameters);
    let mut blob = vec![0u8; unsafe { ffi::ss_phase1_pairs_size(E::CURVE_ID) }];
    let seed = rho_seed();
    let (nc_ptr, nc_len) = match new_challenge {
        Some(b) => (b.as_mut_ptr(), b.len()),
        None => (std::ptr::null_mut(), 0),
    };
    check(unsafe {
        ffi::ss_phase1_verification_vectors_shard(
            &p,
            output.as_ptr(),
            output.len(),
            flag(compressed_output),
            nc_ptr,
            nc_len,
            flag(compressed_new_challenge),
            subgroup_mode(subgroup_check_mode),
            ratio_check as c_int,
            seed.as_ptr(),
            blob.as_mut_ptr(),
            shard.0,
            shard.1,
        )
    })?;
    Ok(blob)
}

/// Host-side reduction of SURVEY.md §8e: the sum of the shards' partial (s, sx) is a valid random linear combination.
pub fn reduce_partial_pairs<E: CudaCurve>(partials: &[Vec<u8>]) -> Result<RatioPairs<E>> {
    let n = unsafe { ffi::ss_phase1_pairs_size(E::CURVE_ID) };
    let mut all = Vec::with_capacity(n * partials.len());
    for p in partials {
        assert_eq!(p.len(), n);
        all.extend_from_slice(p);
    }
    let mut out = vec![0u8; n];
    check(unsafe { ffi::ss_phase1_reduce_partial_pairs(E::CURVE_ID, all.as_ptr(), partials.len() as c_int, out.as_mut_ptr()) })?;
    Ok(read_pairs::<E>(&out))
}

/// The ratio half of `Phase1::verification` with its verdict: vectors + check_power_ratios(_g2) of every vector against
/// (tau_g2[0], tau_g2[1]) / (tau_g1[0], tau_g1[1]) read from the response (verification.rs:58-71, accumulator.rs:56-91).
#[allow(clippy::too_many_arguments)]
pub fn phase1_verification_ratios<E: CudaCurve>(
    output: &[u8],
    new_challenge: &mut [u8],
    compressed_output: UseCompression,
    compressed_new_challenge: UseCompression,
    check_output_for_correctness: CheckForCorrectness,
    subgroup_check_mode: SubgroupCheckMode,
    parameters: &Phase1Parameters<E>,
) -> Result<()> {
    let p = params_of(parameters);
    let seed = rho_seed();
    check(unsafe {
        ffi::ss_phase1_verification_ratios(
            &p,
            output.as_ptr(),
            output.len(),
            flag(compressed_output),
            check_mode(check_output_for_correctness),
            new_challenge.as_mut_ptr(),
            new_challenge.len(),
            flag(compressed_new_challenge),
            subgroup_mode(subgroup_check_mode),
            seed.as_ptr(),
        )
    })
}

/// `Groth16Params::new` + `::write` (setup-utils/src/groth16_utils.rs:81-168), the body of prepare_phase2
/// (phase2-cli/src/prepare_phase2.rs:16-70): phase-1 accumulator bytes in, serialized Groth16Params out.
pub fn groth16_params_new<E: CudaCurve>(
    accumulator: &[u8],
    parameters: &Phase1Parameters<E>,
    phase2_size: usize,
    compressed_input: UseCompression,
    compressed_output: UseCompression,
    check_input_for_correctness: CheckForCorrectness,
) -> Result<Vec<u8>> {
    let p = params_of(parameters);
    let (mut domain, mut bytes) = (0u64, 0usize);
    check(unsafe { ffi::ss_groth16_params_size(E::CURVE_ID, phase2_size as u64, flag(compressed_output), &mut domain, &mut bytes) })?;
    let mut out = vec![0u8; bytes];
    check(unsafe {
        ffi::ss_groth16_params_new(
            &p,
            accumulator.as_ptr(),
            accumulator.len(),
            flag(compressed_input),
            check_mode(check_input_for_correctness),
            phase2_size as u64,
            out.as_mut_ptr(),
            out.len(),
            flag(compressed_output),
        )
    })?;
    Ok(out)
}

// ------------------------------------------------------------------------------------------------------------------
// verdicts from pairs, accumulator re-layout, group transforms, QAP rows (SURVEY.md §8f)
// ------------------------------------------------------------------------------------------------------------------

/// `check_power_ratios` / `check_power_ratios_g2` (phase1/src/helpers/accumulator.rs:56-91) of the four vectors from
/// their (s, sx) pairs blob — the whole-response blob or the `ss_phase1_reduce_partial_pairs` of the shards' blobs —
/// against `g1_check = (tau_g1[0], tau_g1[1])` and `g2_check = (tau_g2[0], tau_g2[1])` (verification.rs:58-71), the four
/// pairing checks run on the device.  `Err(VerificationError::InvalidRatio)` names the failing vector.
pub fn check_ratio_pairs<E: CudaCurve>(
    pairs_blob: &[u8],
    g1_check: &(E::G1Affine, E::G1Affine),
    g2_check: &(E::G2Affine, E::G2Affine),
) -> Result<()> {
    assert_eq!(pairs_blob.len(), unsafe { ffi::ss_phase1_pairs_size(E::CURVE_ID) });
    let a = points_bytes(&[g1_check.0, g1_check.1]);
    let b = points_bytes(&[g2_check.0, g2_check.1]);
    check(unsafe { ffi::ss_phase1_check_ratio_pairs(E::CURVE_ID, pairs_blob.as_ptr(), a.as_ptr(), b.as_ptr()) })
}

/// Several `check_same_ratio` (setup-utils/src/helpers.rs:406-424) in one launch; `Err` carries the first failing index
/// in `ss_last_error().index`.
pub fn check_same_ratio_batch<E: CudaCurve>(
    g1: &[(E::G1Affine, E::G1Affine)],
    g2: &[(E::G2Affine, E::G2Affine)],
) -> core::result::Result<(), usize> {
    assert_eq!(g1.len(), g2.len());
    let a: Vec<E::G1Affine> = g1.iter().flat_map(|p| [p.0, p.1]).collect();
    let b: Vec<E::G2Affine> = g2.iter().flat_map(|p| [p.0, p.1]).collect();
    let (ab, bb) = (points_bytes(&a), points_bytes(&b));
    let mut first_bad: c_int = -1;
    let rc = unsafe { ffi::ss_check_same_ratio_batch(E::CURVE_ID, ab.as_ptr(), bb.as_ptr(), g1.len() as c_int, &mut first_bad) };
    match rc {
        0 => Ok(()),
        10 => Err(first_bad as usize),
        _ => {
            check(rc).expect("pairing inputs are canonical points");
            Ok(())
        }
    }
}

/// One iteration of `Phase1::aggregation` (phase1/src/aggregation.rs:11-180): the vectors of the chunk
/// `chunk_parameters.chunk_index` are written into the full accumulator (beta_g2 comes from chunk 0).
pub fn phase1_aggregate_chunk<E: CudaCurve>(
    chunk: &[u8],
    compressed_chunk: UseCompression,
    full: &mut [u8],
    compressed_full: UseCompression,
    chunk_parameters: &Phase1Parameters<E>,
) -> Result<()> {
    let p = params_of(chunk_parameters);
    check(unsafe {
        ffi::ss_phase1_aggregate_chunk(&p, chunk.as_ptr(), chunk.len(), flag(compressed_chunk), full.as_mut_ptr(), full.len(), flag(compressed_full))
    })
}

/// One iteration of `Phase1::split` (phase1/src/aggregation.rs:189-353): the reverse of `phase1_aggregate_chunk`.
pub fn phase1_split_chunk<E: CudaCurve>(
    full: &[u8],
    compressed_full: UseCompression,
    chunk: &mut [u8],
    compressed_chunk: UseCompression,
    chunk_parameters: &Phase1Parameters<E>,
) -> Result<()> {
    let p = params_of(chunk_parameters);
    check(unsafe {
        ffi::ss_phase1_split_chunk(&p, full.as_ptr(), full.len(), flag(compressed_full), chunk.as_mut_ptr(), chunk.len(), flag(compressed_chunk))
    })
}

/// `helpers::accumulator::decompress` (phase1/src/helpers/accumulator.rs:200-301): compressed accumulator ->
/// uncompressed, elements read with `check_input_for_correctness`.
pub fn phase1_decompress<E: CudaCurve>(
    input: &[u8],
    output: &mut [u8],
    check_input_for_correctness: CheckForCorrectness,
    parameters: &Phase1Parameters<E>,
) -> Result<()> {
    let p = params_of(parameters);
    check(unsafe {
        ffi::ss_phase1_decompress(&p, input.as_ptr(), input.len(), check_mode(check_input_for_correctness), output.as_mut_ptr(), output.len())
    })
}

/// `to_coeffs` = `domain.ifft` over curve points (setup-utils/src/groth16_utils.rs:44-53); `n` a power of two.
pub fn group_ifft<C: CudaGroup>(points: &[C]) -> Result<Vec<C>> {
    let input = points_bytes(points);
    let mut out = vec![0u8; input.len()];
    check(unsafe {
        ffi::ss_group_ifft(C::CURVE_ID, C::GROUP_ID, input.as_ptr(), 0, check_mode(CheckForCorrectness::No), points.len(), out.as_mut_ptr(), 0)
    })?;
    Ok(read_points::<C>(&out, points.len()))
}

/// `h_query_groth16` (setup-utils/src/groth16_utils.rs:59-63): out_i = powers[i + degree] - powers[i], i < degree - 1.
pub fn h_query_groth16<C: CudaGroup>(powers: &[C], degree: usize) -> Result<Vec<C>> {
    let input = points_bytes(powers);
    let n_out = degree.saturating_sub(1);
    let mut out = vec![0u8; n_out * C::zero().uncompressed_size()];
    check(unsafe {
        ffi::ss_h_query_groth16(C::CURVE_ID, input.as_ptr(), 0, check_mode(CheckForCorrectness::No), powers.len(), degree, out.as_mut_ptr(), 0)
    })?;
    Ok(read_points::<C>(&out, n_out))
}

/// `dot_product_vec` + `normalize_batch` (phase2/src/polynomial.rs:30-47,75-94): one point per CSR row,
/// out_v = sum over the row's entries of coeffs[e] * bases[index[e]].
pub fn qap_dot_product<C: CudaGroup>(
    bases: &[C],
    row_ptr: &[u64],
    index: &[u32],
    coeffs: &[C::ScalarField],
) -> Result<Vec<C>> {
    assert!(!row_ptr.is_empty() && index.len() == coeffs.len() && *row_ptr.last().unwrap() as usize == index.len());
    let rows = row_ptr.len() - 1;
    let (bb, cb) = (points_bytes(bases), scalars_bytes(coeffs));
    let mut out = vec![0u8; rows * C::zero().uncompressed_size()];
    check(unsafe {
        ffi::ss_qap_dot_product(
            C::CURVE_ID,
            C::GROUP_ID,
            bb.as_ptr(),
            0,
            check_mode(CheckForCorrectness::No),
            bases.len(),
            row_ptr.as_ptr(),
            index.as_ptr(),
            cb.as_ptr(),
            rows,
            out.as_mut_ptr(),
            0,
        )
    })?;
    Ok(read_points::<C>(&out, rows))
}

// ------------------------------------------------------------------------------------------------------------------
// phase 2: MPCParameters::contribute / verify on the H and L queries (SURVEY.md config C5)
// ------------------------------------------------------------------------------------------------------------------

fn g1_size<E: CudaCurve>(compression: UseCompression) -> usize {
    match compression {
        Compress::Yes => E::G1Affine::zero().compressed_size(),
        Compress::No => E::G1Affine::zero().uncompressed_size(),
    }
}

/// The hot half of `MPCParameters::contribute` (phase2/src/parameters.rs:286-307; streaming twin
/// chunked_groth16.rs:387-466): every element of the serialized `h_query` / `l_query` <- delta^-1 * element and
/// `delta_g1` / `delta_g2` <- delta * element, in place, all serialized with `compression` and read with
/// `check_input_for_correctness`.  `shard = (index, count)` processes that index-range part of each query only
/// (`(0, 1)`: whole queries); delta_g1 / delta_g2 belong to shard 0.
pub fn phase2_contribute<E: CudaCurve>(
    h_query: &mut [u8],
    l_query: &mut [u8],
    delta_g1: Option<&mut [u8]>,
    delta_g2: Option<&mut [u8]>,
    delta: &E::ScalarField,
    compression: UseCompression,
    check_input_for_correctness: CheckForCorrectness,
    shard: (u32, u32),
) -> Result<()> {
    let size = g1_size::<E>(compression);
    let d = scalar_bytes(delta);
    let p1 = delta_g1.map_or(core::ptr::null_mut(), |b| b.as_mut_ptr());
    let p2 = delta_g2.map_or(core::ptr::null_mut(), |b| b.as_mut_ptr());
    check(unsafe {
        ffi::ss_phase2_contribute_shard(
            E::CURVE_ID,
            d.as_ptr(),
            h_query.as_mut_ptr(),
            h_query.len() / size,
            l_query.as_mut_ptr(),
            l_query.len() / size,
            flag(compression),
            check_mode(check_input_for_correctness),
            p1,
            p2,
            shard.0,
            shard.1,
        )
    })
}

/// `merge_pairs(before.h, after.h)` and `merge_pairs(before.l, after.l)` of MPCParameters::verify
/// (phase2/src/parameters.rs:393-407) over shard `shard` of the serialized queries, with read_groth16_fast's subgroup
/// check on `after` (:566-581): the pairs blob (s_h, sx_h, s_l, sx_l), partial sums for a shard.
pub fn phase2_verification_pairs<E: CudaCurve>(
    before: (&[u8], &[u8]),
    after: (&[u8], &[u8]),
    compression: UseCompression,
    check_before: CheckForCorrectness,
    check_after: CheckForCorrectness,
    subgroup_check_mode: SubgroupCheckMode,
    shard: (u32, u32),
) -> Result<Vec<u8>> {
    let size = g1_size::<E>(compression);
    assert!(before.0.len() == after.0.len() && before.1.len() == after.1.len());
    let seed = rho_seed();
    let mut pairs = vec![0u8; unsafe { ffi::ss_phase2_pairs_size(E::CURVE_ID) }];
    check(unsafe {
        ffi::ss_phase2_verification_pairs(
            E::CURVE_ID,
            before.0.as_ptr(),
            after.0.as_ptr(),
            before.0.len() / size,
            before.1.as_ptr(),
            after.1.as_ptr(),
            before.1.len() / size,
            flag(compression),
            check_mode(check_before),
            check_mode(check_after),
            subgroup_mode(subgroup_check_mode),
            seed.as_ptr(),
            pairs.as_mut_ptr(),
            shard.0,
            shard.1,
        )
    })?;
    Ok(pairs)
}

/// Element-wise sums of the shards' phase-2 pairs blobs.
pub fn phase2_reduce_partial_pairs<E: CudaCurve>(blobs: &[Vec<u8>]) -> Result<Vec<u8>> {
    let size = unsafe { ffi::ss_phase2_pairs_size(E::CURVE_ID) };
    assert!(blobs.iter().all(|b| b.len() == size));
    let all: Vec<u8> = blobs.concat();
    let mut pairs = vec![0u8; size];
    check(unsafe { ffi::ss_phase2_reduce_partial_pairs(E::CURVE_ID, all.as_ptr(), blobs.len() as c_int, pairs.as_mut_ptr()) })?;
    Ok(pairs)
}

/// The ratio checks of MPCParameters::verify from a (reduced) pairs blob, on the device: 0 = delta_g1 / delta_g2
/// consistency, 1 = H, 2 = L (parameters.rs:393-407) — `ss_last_error().index` names the failing one.
pub fn phase2_check_ratio_pairs<E: CudaCurve>(
    pairs_blob: &[u8],
    delta_g1_after: &E::G1Affine,
    delta_g2_before: &E::G2Affine,
    delta_g2_after: &E::G2Affine,
) -> Result<()> {
    assert_eq!(pairs_blob.len(), unsafe { ffi::ss_phase2_pairs_size(E::CURVE_ID) });
    let d1 = points_bytes(&[*delta_g1_after]);
    let (d2b, d2a) = (points_bytes(&[*delta_g2_before]), points_bytes(&[*delta_g2_after]));
    check(unsafe { ffi::ss_phase2_check_ratio_pairs(E::CURVE_ID, pairs_blob.as_ptr(), d1.as_ptr(), d2b.as_ptr(), d2a.as_ptr()) })
}

/// The H / L queries and delta checks of MPCParameters::verify (phase2/src/parameters.rs:314-411) in one call: queries
/// and the three delta elements serialized with `compression`.  The byte comparisons of the unchanged parts and the
/// proof-of-knowledge / transcript checks stay with the caller.
pub fn phase2_verify<E: CudaCurve>(
    before: (&[u8], &[u8]),
    after: (&[u8], &[u8]),
    delta_g1_after: &[u8],
    delta_g2_before: &[u8],
    delta_g2_after: &[u8],
    compression: UseCompression,
    check_before: CheckForCorrectness,
    check_after: CheckForCorrectness,
    subgroup_check_mode: SubgroupCheckMode,
) -> Result<()> {
    let size = g1_size::<E>(compression);
    assert!(before.0.len() == after.0.len() && before.1.len() == after.1.len());
    let seed = rho_seed();
    check(unsafe {
        ffi::ss_phase2_verification(
            E::CURVE_ID,
            before.0.as_ptr(),
            after.0.as_ptr(),
            before.0.len() / size,
            before.1.as_ptr(),
            after.1.as_ptr(),
            before.1.len() / size,
            flag(compression),
            check_mode(check_before),
            check_mode(check_after),
            subgroup_mode(subgroup_check_mode),
            delta_g1_after.as_ptr(),
            delta_g2_before.as_ptr(),
            delta_g2_after.as_ptr(),
            seed.as_ptr(),
        )
    })
}
