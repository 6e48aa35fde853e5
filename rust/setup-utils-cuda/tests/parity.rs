//! Parity of the CUDA engine with the reference's own arkworks path: same seeded inputs through both, bytes compared.
//! Run with `SNARK_SETUP_B200_DIR=<checkout> cargo test -p setup-utils-cuda -- --test-threads 1` on a box with a B200.
//! These tests are what turns the repository's "parity asserted by construction" into "parity pinned against the Rust
//! binary" (DESIGN.md §5): they pin the ark-serialize layout, the generator constants and the FFT domain generator.
use ark_bls12_377::Bls12_377;
use ark_ec::pairing::Pairing;
use phase1::{helpers::testing::{generate_input, generate_output}, Phase1, Phase1Parameters, ProvingSystem};
use setup_utils::{
    calculate_hash, derive_rng_from_seed, same_ratio, BatchExpMode, CheckForCorrectness, Groth16Params, SubgroupCheckMode,
    UseCompression,
};

#[test]
fn cuda_matches_arkworks_phase1_bls12_377() {
    let params = Phase1Parameters::<Bls12_377>::new_full(ProvingSystem::Groth16, 10, 256);
    let (input, _) = generate_input(&params, UseCompression::No);
    let mut rng = derive_rng_from_seed(b"parity");
    let (pubkey, privkey) = Phase1::key_generation(&mut rng, &[0u8; 64]).unwrap();

    // contribute: response bytes and therefore the .hash file
    let mut cpu = generate_output(&params, UseCompression::Yes);
    Phase1::computation(&input, &mut cpu, UseCompression::No, UseCompression::Yes, CheckForCorrectness::No, BatchExpMode::Auto, &privkey, &params)
        .unwrap();
    let mut gpu = generate_output(&params, UseCompression::Yes);
    setup_utils_cuda::phase1_computation(&input, &mut gpu, UseCompression::No, UseCompression::Yes, CheckForCorrectness::No, BatchExpMode::Auto, &privkey, &params)
        .unwrap();
    assert_eq!(cpu, gpu);
    assert_eq!(calculate_hash(&cpu), calculate_hash(&gpu));

    // the same computation as two index-range shards writing into one buffer
    let mut sharded = generate_output(&params, UseCompression::Yes);
    for r in 0..2 {
        setup_utils_cuda::phase1_computation_shard(&input, &mut sharded, UseCompression::No, UseCompression::Yes, CheckForCorrectness::No, &privkey, &params, (r, 2))
            .unwrap();
    }
    assert_eq!(cpu, sharded);

    // verify: the new challenge the reference writes, and the four ratio verdicts
    let mut nc_cpu = generate_output(&params, UseCompression::No);
    Phase1::verification(
        &input, &cpu, &mut nc_cpu, &pubkey, &[0u8; 64], UseCompression::No, UseCompression::Yes, UseCompression::No,
        CheckForCorrectness::No, CheckForCorrectness::Full, SubgroupCheckMode::Auto, true, &params,
    )
    .unwrap();
    let mut nc_gpu = generate_output(&params, UseCompression::No);
    setup_utils_cuda::phase1_verification_ratios(
        &gpu, &mut nc_gpu, UseCompression::Yes, UseCompression::No, CheckForCorrectness::Full, SubgroupCheckMode::Auto, &params,
    )
    .unwrap();
    assert_eq!(nc_cpu[64..], nc_gpu[64..]); // the hash prefix is the caller's

    // a tampered response is rejected by both
    let mut bad = gpu.clone();
    let g1c = params.curve.g1_compressed_size;
    let (a, b) = (64 + 5 * g1c, 64 + 6 * g1c);
    let tmp = bad[a..a + g1c].to_vec();
    bad.copy_within(b..b + g1c, a);
    bad[b..b + g1c].copy_from_slice(&tmp);
    assert!(setup_utils_cuda::phase1_verification_ratios(
        &bad, &mut nc_gpu, UseCompression::Yes, UseCompression::No, CheckForCorrectness::Full, SubgroupCheckMode::Auto, &params
    )
    .is_err());
}

#[test]
fn cuda_matches_arkworks_prepare_phase2_and_ratio() {
    let params = Phase1Parameters::<Bls12_377>::new_full(ProvingSystem::Groth16, 10, 256);
    let (input, _) = generate_input(&params, UseCompression::No);
    let mut rng = derive_rng_from_seed(b"parity-2");
    let (_, privkey) = Phase1::key_generation(&mut rng, &[0u8; 64]).unwrap();
    let mut accumulator = generate_output(&params, UseCompression::No);
    Phase1::computation(&input, &mut accumulator, UseCompression::No, UseCompression::No, CheckForCorrectness::No, BatchExpMode::Auto, &privkey, &params)
        .unwrap();
    let acc = Phase1::deserialize(&accumulator, UseCompression::No, CheckForCorrectness::No, &params).unwrap();
    let cpu = Groth16Params::<Bls12_377>::new(
        1 << 10,
        acc.tau_powers_g1.clone(),
        acc.tau_powers_g2.clone(),
        acc.alpha_tau_powers_g1.clone(),
        acc.beta_tau_powers_g1.clone(),
        acc.beta_g2,
    )
    .unwrap();
    let mut want = vec![];
    cpu.write(&mut want, UseCompression::No).unwrap();
    let got = setup_utils_cuda::groth16_params_new(&accumulator, &params, 1 << 10, UseCompression::No, UseCompression::No, CheckForCorrectness::No).unwrap();
    assert_eq!(want, got); // Lagrange coefficients (pins the FFT domain generator) + H query, byte for byte

    let g1 = (acc.tau_powers_g1[0], acc.tau_powers_g1[1]);
    let g2 = (acc.tau_powers_g2[0], acc.tau_powers_g2[1]);
    assert_eq!(same_ratio::<Bls12_377>(&g1, &g2), setup_utils_cuda::same_ratio::<Bls12_377>(&g1, &g2));
    let bad = (acc.tau_powers_g2[0], acc.tau_powers_g2[2]);
    assert_eq!(same_ratio::<Bls12_377>(&g1, &bad), setup_utils_cuda::same_ratio::<Bls12_377>(&g1, &bad));
    let _ = <Bls12_377 as Pairing>::G1Affine::default();
}

#[test]
fn cuda_helpers_match_setup_utils() {
    use ark_bls12_377::{Fr, G1Affine, G2Affine};
    use ark_ec::{AffineRepr, CurveGroup};
    use ark_ff::UniformRand;
    let mut rng = derive_rng_from_seed(b"parity-3");
    let n = 300;
    let exps: Vec<Fr> = (0..n).map(|_| Fr::rand(&mut rng)).collect();
    let coeff = Fr::rand(&mut rng);
    let bases1: Vec<G1Affine> = (0..n).map(|_| (G1Affine::generator() * Fr::rand(&mut rng)).into_affine()).collect();
    let bases2: Vec<G2Affine> = (0..n).map(|_| (G2Affine::generator() * Fr::rand(&mut rng)).into_affine()).collect();
    let (mut a, mut b) = (bases1.clone(), bases1.clone());
    setup_utils::batch_exp(&mut a, &exps, Some(&coeff), BatchExpMode::Auto).unwrap();
    setup_utils_cuda::batch_exp(&mut b, &exps, Some(&coeff), BatchExpMode::Auto).unwrap();
    assert_eq!(a, b);
    let (mut a, mut b) = (bases2.clone(), bases2.clone());
    setup_utils::batch_mul(&mut a, &coeff, BatchExpMode::Auto).unwrap();
    setup_utils_cuda::batch_mul(&mut b, &coeff, BatchExpMode::Auto).unwrap();
    assert_eq!(a, b);
    assert_eq!(
        setup_utils::generate_powers_of_tau::<Bls12_377>(&coeff, 5, 40),
        setup_utils_cuda::generate_powers_of_tau::<Bls12_377>(&coeff, 5, 40)
    );
    // power_pairs uses fresh randomness on both sides: compare the verdicts, not the points
    let tau = Fr::rand(&mut rng);
    let mut v = vec![G1Affine::generator(); 64];
    let powers = setup_utils::generate_powers_of_tau::<Bls12_377>(&tau, 0, 64);
    setup_utils::batch_exp(&mut v, &powers, None, BatchExpMode::Auto).unwrap();
    let gx = (G2Affine::generator() * tau).into_affine();
    assert!(same_ratio::<Bls12_377>(&setup_utils_cuda::power_pairs(&v), &(G2Affine::generator(), gx)));
    v[7] = (v[7] * Fr::rand(&mut rng)).into_affine();
    assert!(!same_ratio::<Bls12_377>(&setup_utils_cuda::power_pairs(&v), &(G2Affine::generator(), gx)));
    assert!(setup_utils_cuda::check_subgroup(&bases1, SubgroupCheckMode::Auto).is_ok());
}

/// The sharded verification loop: three index-range shards of one response, partial pairs added, verdict from the pairs
/// — and the re-layout wrappers against the reference's `decompress`.
#[test]
fn cuda_sharded_verification_and_relayout() {
    let params = Phase1Parameters::<Bls12_377>::new_full(ProvingSystem::Groth16, 8, 64);
    let (input, _) = generate_input(&params, UseCompression::No);
    let mut rng = derive_rng_from_seed(b"parity-4");
    let (_, privkey) = Phase1::key_generation(&mut rng, &[0u8; 64]).unwrap();
    let mut response = generate_output(&params, UseCompression::Yes);
    Phase1::computation(&input, &mut response, UseCompression::No, UseCompression::Yes, CheckForCorrectness::No, BatchExpMode::Auto, &privkey, &params)
        .unwrap();
    let n_resp = response.len() - params.public_key_size;
    let mut new_challenge = vec![0u8; params.accumulator_size];
    let blobs: Vec<Vec<u8>> = (0..3u32)
        .map(|s| {
            setup_utils_cuda::phase1_verification_vectors_shard(
                &response[..n_resp], Some(&mut new_challenge[..]), UseCompression::Yes, UseCompression::No, SubgroupCheckMode::Auto, true, &params, (s, 3),
            )
            .unwrap()
        })
        .collect();
    let pairs = setup_utils_cuda::reduce_partial_pairs::<Bls12_377>(&blobs).unwrap();
    let acc = Phase1::deserialize(&response[..n_resp], UseCompression::Yes, CheckForCorrectness::Full, &params).unwrap();
    let g1 = (acc.tau_powers_g1[0], acc.tau_powers_g1[1]);
    let g2 = (acc.tau_powers_g2[0], acc.tau_powers_g2[1]);
    assert!(same_ratio::<Bls12_377>(&pairs.tau_g1, &g2));
    assert!(same_ratio::<Bls12_377>(&g1, &pairs.tau_g2));
    assert!(same_ratio::<Bls12_377>(&pairs.alpha_g1, &g2));
    assert!(same_ratio::<Bls12_377>(&pairs.beta_g1, &g2));
    // the new challenge the shards wrote is the reference's decompressed response
    let mut want = vec![0u8; params.accumulator_size];
    phase1::helpers::accumulator::decompress(&response[..n_resp], &mut want, CheckForCorrectness::No, &params).unwrap();
    assert_eq!(want[64..], new_challenge[64..]);
    let mut got = vec![0u8; params.accumulator_size];
    setup_utils_cuda::phase1_decompress(&response[..n_resp], &mut got, CheckForCorrectness::No, &params).unwrap();
    assert_eq!(want[64..], got[64..]);
}

/// Phase 2: `MPCParameters::contribute` updates delta_g1 / delta_g2 by delta and the H and L queries by delta^-1
/// (phase2/src/parameters.rs:286-307), and `verify` checks them with merge_pairs + same_ratio (:393-407).  Building
/// MPCParameters needs a circuit, so the reference side here is that body through setup_utils (batch_mul, merge_pairs,
/// same_ratio) on compressed query bytes; the engine side is one call each way, whole and as three shards.
#[test]
fn cuda_phase2_contribute_and_verify_match_setup_utils() {
    use ark_bls12_377::{Fr, G1Affine, G2Affine};
    use ark_ec::{AffineRepr, CurveGroup};
    use ark_ff::{Field, UniformRand};
    use ark_serialize::{CanonicalDeserialize, CanonicalSerialize};
    let mut rng = derive_rng_from_seed(b"parity-5");
    let (nh, nl) = (255, 256);
    let pts = |n: usize, rng: &mut _| -> Vec<G1Affine> { (0..n).map(|_| (G1Affine::generator() * Fr::rand(rng)).into_affine()).collect() };
    let (h, l) = (pts(nh, &mut rng), pts(nl, &mut rng));
    let ser = |v: &[G1Affine]| -> Vec<u8> {
        let mut b = Vec::new();
        for p in v {
            p.serialize_compressed(&mut b).unwrap();
        }
        b
    };
    let delta = Fr::rand(&mut rng);
    let d1_before = (G1Affine::generator() * Fr::rand(&mut rng)).into_affine();
    let d2_before = (G2Affine::generator() * Fr::rand(&mut rng)).into_affine();

    // reference body: delta_g1 *= delta, delta_g2 *= delta, queries batch_mul'd by delta^-1
    let (mut h_ref, mut l_ref) = (h.clone(), l.clone());
    let inv = delta.inverse().unwrap();
    setup_utils::batch_mul(&mut h_ref, &inv, BatchExpMode::Auto).unwrap();
    setup_utils::batch_mul(&mut l_ref, &inv, BatchExpMode::Auto).unwrap();
    let d1_after = (d1_before * delta).into_affine();
    let d2_after = (d2_before * delta).into_affine();

    let (mut hb, mut lb) = (ser(&h), ser(&l));
    let mut d1b = ser(&[d1_before]);
    let mut d2b = Vec::new();
    d2_before.serialize_compressed(&mut d2b).unwrap();
    let d2_before_bytes = d2b.clone();
    setup_utils_cuda::phase2_contribute::<Bls12_377>(
        &mut hb, &mut lb, Some(&mut d1b), Some(&mut d2b), &delta, UseCompression::Yes, CheckForCorrectness::Full, (0, 1),
    )
    .unwrap();
    assert_eq!(hb, ser(&h_ref));
    assert_eq!(lb, ser(&l_ref));
    assert_eq!(G1Affine::deserialize_compressed(&d1b[..]).unwrap(), d1_after);
    assert_eq!(G2Affine::deserialize_compressed(&d2b[..]).unwrap(), d2_after);

    // three shards into one pair of buffers give the same bytes
    let (mut hs, mut ls) = (ser(&h), ser(&l));
    for s in 0..3u32 {
        setup_utils_cuda::phase2_contribute::<Bls12_377>(&mut hs, &mut ls, None, None, &delta, UseCompression::Yes, CheckForCorrectness::No, (s, 3))
            .unwrap();
    }
    assert_eq!((hs, ls), (hb.clone(), lb.clone()));

    // verify: the reference's verdict on the engine's output, and the engine's verdict
    let g2_pair = (d2_after, d2_before);
    assert!(same_ratio::<Bls12_377>(&setup_utils::merge_pairs(&h, &h_ref), &g2_pair));
    assert!(same_ratio::<Bls12_377>(&setup_utils::merge_pairs(&l, &l_ref), &g2_pair));
    let (h0, l0) = (ser(&h), ser(&l));
    setup_utils_cuda::phase2_verify::<Bls12_377>(
        (&h0, &l0), (&hb, &lb), &d1b, &d2_before_bytes, &d2b, UseCompression::Yes, CheckForCorrectness::No,
        CheckForCorrectness::OnlyNonZero, SubgroupCheckMode::Auto,
    )
    .unwrap();
    let blobs: Vec<Vec<u8>> = (0..3u32)
        .map(|s| {
            setup_utils_cuda::phase2_verification_pairs::<Bls12_377>(
                (&h0, &l0), (&hb, &lb), UseCompression::Yes, CheckForCorrectness::No, CheckForCorrectness::OnlyNonZero,
                SubgroupCheckMode::Auto, (s, 3),
            )
            .unwrap()
        })
        .collect();
    let pairs = setup_utils_cuda::phase2_reduce_partial_pairs::<Bls12_377>(&blobs).unwrap();
    setup_utils_cuda::phase2_check_ratio_pairs::<Bls12_377>(&pairs, &d1_after, &d2_before, &d2_after).unwrap();
    // an H element replaced by its neighbour is rejected by both
    let g1c = 48;
    let mut bad = hb.clone();
    bad.copy_within(g1c..2 * g1c, 0);
    assert!(setup_utils_cuda::phase2_verify::<Bls12_377>(
        (&h0, &l0), (&bad, &lb), &d1b, &d2_before_bytes, &d2b, UseCompression::Yes, CheckForCorrectness::No,
        CheckForCorrectness::OnlyNonZero, SubgroupCheckMode::Auto,
    )
    .is_err());
    let mut h_bad = h_ref.clone();
    h_bad[0] = h_bad[1];
    assert!(!same_ratio::<Bls12_377>(&setup_utils::merge_pairs(&h, &h_bad), &g2_pair));
}
