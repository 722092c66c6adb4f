//! Drop-in for the arkworks calls on the reference's prove path, backed by libb200zk (sm_100a CUDA).
//!
//! | arkworks item (reference call site)                                                       | here |
//! |---|---|
//! | `Groth16::<Bls12_381>::prove` (fibbonaci_handler.rs:110, matrix_proof.rs:139-140, prime_snark.rs:119) | [`B200Groth16::prove`] |
//! | `LibsnarkReduction::witness_map_from_matrices` (`R1CSToQAP`)                               | [`B200Reduction`] |
//! | `VariableBaseMSM::msm_bigint` for G1 / G2                                                  | [`msm_bigint_g1`], [`msm_bigint_g2`] |
//! | `Radix2EvaluationDomain::{fft,ifft}_in_place`, `get_coset`                                | [`ntt_in_place`] |
//! | `prepare_verifying_key` + `serialize_compressed` (matrix_proof.rs:134-136, io.rs:62-68)    | [`prepared_vk_bytes`] |
//! | `Groth16::verify_with_processed_vk` (matrix_proof.rs:199-206)                              | [`verify_with_processed_vk`] |
//! | the same for many proofs against one pvk, on the GPU, one verdict per proof                | [`verify_batch_with_processed_vk`] |
//! | `Groth16::<Bls12_381>::setup` (matrix_proof.rs:128-131, fibbonaci_handler.rs:107)          | [`DeviceKey::setup`] |
//!
//! SOURCE ONLY -- never compiled in the build image (no Rust toolchain there).  arkworks' `Fp` / `Affine` are
//! `repr(Rust)`: limbs are copied explicitly (`x.0 .0`), never transmuted.  Field elements cross in Montgomery form
//! (arkworks' in-memory form), MSM scalars as `into_bigint()`.
#![allow(non_camel_case_types, clippy::missing_safety_doc)]

use ark_bls12_381::{Bls12_381, Fr, G1Affine, G1Projective, G2Affine, G2Projective};
use ark_ec::AffineRepr;
use ark_ff::{BigInt, Field, PrimeField, Zero};
use ark_groth16::{r1cs_to_qap::R1CSToQAP, Proof, ProvingKey, VerifyingKey};
use ark_poly::EvaluationDomain;
use ark_relations::r1cs::{
    ConstraintMatrices, ConstraintSynthesizer, ConstraintSystem, ConstraintSystemRef, OptimizationGoal, SynthesisError,
};
use ark_serialize::CanonicalDeserialize;
use ark_std::{rand::RngCore, UniformRand};
use std::{ffi::CStr, os::raw::c_char, ptr};

/// Raw bindings: `bindgen include/b200zk.h`, written out by hand.
pub mod sys {
    use super::c_char;
    #[repr(C)] pub struct b2z_ctx { _p: [u8; 0] }
    #[repr(C)] pub struct b2z_pk { _p: [u8; 0] }
    #[repr(C)] pub struct b2z_r1cs { _p: [u8; 0] }
    #[repr(C)]
    pub struct b2z_pk_desc {
        pub num_variables: u64, pub num_instance: u64, pub log_domain: u32,
        pub a_query: *const u64, pub a_inf: *const u8,
        pub b_g1_query: *const u64, pub b_g1_inf: *const u8,
        pub b_g2_query: *const u64, pub b_g2_inf: *const u8,
        pub h_query: *const u64, pub h_inf: *const u8,
        pub l_query: *const u64, pub l_inf: *const u8,
        pub alpha_g1: *const u64, pub beta_g1: *const u64, pub delta_g1: *const u64,
        pub beta_g2: *const u64, pub delta_g2: *const u64,
    }
    #[repr(C)]
    pub struct b2z_setup_desc {
        pub alpha: *const u64, pub beta: *const u64, pub gamma: *const u64, pub delta: *const u64, pub tau: *const u64,
        pub g1_generator: *const u64, pub g2_generator: *const u64,
    }
    #[repr(C)]
    pub struct b2z_vk_out {
        pub alpha_g1: [u64; 12], pub beta_g2: [u64; 24], pub gamma_g2: [u64; 24], pub delta_g2: [u64; 24],
        pub gamma_abc_g1: *mut u64, pub gamma_abc_inf: *mut u8,
    }
    #[repr(C)]
    pub struct b2z_vk_desc {
        pub num_instance: u64,
        pub alpha_g1: *const u64, pub beta_g2: *const u64, pub gamma_g2: *const u64, pub delta_g2: *const u64,
        pub gamma_abc_g1: *const u64, pub gamma_abc_inf: *const u8,
    }
    pub const B2Z_OK: i32 = 0;
    pub const B2Z_EINVAL: i32 = 1;
    pub const B2Z_ESIZE: i32 = 2;
    pub const B2Z_PARTIAL_BYTES: usize = 1344;
    extern "C" {
        pub fn b2z_ctx_create(device_id: i32, out: *mut *mut b2z_ctx) -> i32;
        pub fn b2z_ctx_destroy(ctx: *mut b2z_ctx);
        pub fn b2z_groth16_setup(ctx: *mut b2z_ctx, r1cs: *mut b2z_r1cs, desc: *const b2z_setup_desc,
                                 pk_out: *mut *mut b2z_pk, vk_out: *mut b2z_vk_out) -> i32;
        pub fn b2z_groth16_setup_shard(ctx: *mut b2z_ctx, r1cs: *mut b2z_r1cs, desc: *const b2z_setup_desc, rank: u32,
                                       world: u32, pk_out: *mut *mut b2z_pk, vk_out: *mut b2z_vk_out) -> i32;
        pub fn b2z_last_error(ctx: *const b2z_ctx) -> *const c_char;
        pub fn b2z_ntt_fr(ctx: *mut b2z_ctx, data: *mut u64, log_n: u32, inverse: i32, coset_gen: *const u64) -> i32;
        pub fn b2z_witness_map(ctx: *mut b2z_ctx, a: *const u64, b: *const u64, c: *const u64, log_n: u32, h: *mut u64) -> i32;
        pub fn b2z_msm_g1(ctx: *mut b2z_ctx, bases: *const u64, inf: *const u8, scalars: *const u64, n: u64, out: *mut u64) -> i32;
        pub fn b2z_msm_g2(ctx: *mut b2z_ctx, bases: *const u64, inf: *const u8, scalars: *const u64, n: u64, out: *mut u64) -> i32;
        pub fn b2z_pk_upload(ctx: *mut b2z_ctx, desc: *const b2z_pk_desc, out: *mut *mut b2z_pk) -> i32;
        pub fn b2z_pk_upload_shard(ctx: *mut b2z_ctx, desc: *const b2z_pk_desc, rank: u32, world: u32, out: *mut *mut b2z_pk) -> i32;
        pub fn b2z_pk_free(ctx: *mut b2z_ctx, pk: *mut b2z_pk);
        pub fn b2z_groth16_prove(ctx: *mut b2z_ctx, pk: *const b2z_pk, a: *const u64, b: *const u64, c: *const u64,
                                 z: *const u64, r: *const u64, s: *const u64, proof_out: *mut u8) -> i32;
        pub fn b2z_r1cs_upload(ctx: *mut b2z_ctx, num_constraints: u64, num_instance: u64, num_variables: u64,
                               a_row_ptr: *const u64, a_cols: *const u32, a_coeffs: *const u64,
                               b_row_ptr: *const u64, b_cols: *const u32, b_coeffs: *const u64,
                               c_row_ptr: *const u64, c_cols: *const u32, c_coeffs: *const u64, out: *mut *mut b2z_r1cs) -> i32;
        pub fn b2z_r1cs_free(ctx: *mut b2z_ctx, r1cs: *mut b2z_r1cs);
        pub fn b2z_witness_map_from_matrices(ctx: *mut b2z_ctx, r1cs: *mut b2z_r1cs, z: *const u64, h_out: *mut u64) -> i32;
        pub fn b2z_groth16_prove_r1cs(ctx: *mut b2z_ctx, pk: *const b2z_pk, r1cs: *mut b2z_r1cs, z: *const u64,
                                      r: *const u64, s: *const u64, proof_out: *mut u8) -> i32;
        pub fn b2z_groth16_prove_partial_r1cs(ctx: *mut b2z_ctx, pk: *const b2z_pk, r1cs: *mut b2z_r1cs, z: *const u64,
                                              r: *const u64, s: *const u64, partial_out: *mut u8) -> i32;
        pub fn b2z_groth16_combine(partials: *const u8, world: u32, proof_out: *mut u8) -> i32;
        pub fn b2z_host_register(ctx: *mut b2z_ctx, ptr: *mut std::ffi::c_void, bytes: u64) -> i32;
        pub fn b2z_host_unregister(ctx: *mut b2z_ctx, ptr: *mut std::ffi::c_void) -> i32;
        pub fn b2z_groth16_prepare_verifying_key(vk: *const b2z_vk_desc, pvk_out: *mut u8, capacity: u64, pvk_len: *mut u64) -> i32;
        pub fn b2z_groth16_verify_with_processed_vk(pvk: *const u8, pvk_len: u64, public_inputs: *const u64, num_inputs: u64,
                                                    proof: *const u8, valid: *mut i32) -> i32;
        pub fn b2z_groth16_verify_batch(ctx: *mut b2z_ctx, pvk: *const u8, pvk_len: u64, public_inputs: *const u64,
                                        num_inputs: u64, proofs: *const u8, count: u64, results: *mut i32) -> i32;
        // key-generation scalars on the host cores (no ctx): see INTEGRATION.md section 7
        pub fn b2z_fr_lagrange_at(log_n: u32, tau: *const u64, count: u64, threads: u32, out: *mut u64) -> i32;
        pub fn b2z_fr_geometric(base: *const u64, scale: *const u64, count: u64, threads: u32, out: *mut u64) -> i32;
        pub fn b2z_fr_lincomb3(count: u64, a: *const u64, x: *const u64, b: *const u64, y: *const u64, c: *const u64,
                               z: *const u64, threads: u32, out: *mut u64) -> i32;
        pub fn b2z_fr_into_bigint(count: u64, input: *const u64, threads: u32, out: *mut u64) -> i32;
        pub fn b2z_spmv_fr(ctx: *mut b2z_ctx, nrows: u64, ncols: u64, row_ptr: *const u64, cols: *const u32,
                           coeffs: *const u64, x: *const u64, y_out: *mut u64) -> i32;
        pub fn b2z_fixed_base_mul_g1(ctx: *mut b2z_ctx, scalars: *const u64, n: u64, out_points: *mut u64, out_inf: *mut u8) -> i32;
        pub fn b2z_fixed_base_mul_g2(ctx: *mut b2z_ctx, scalars: *const u64, n: u64, out_points: *mut u64, out_inf: *mut u8) -> i32;
        // host-side witness helpers (no ctx): Poseidon digest with the caller's PoseidonConfig, modpow tables
        pub fn b2z_poseidon_hash(params: *const b2z_poseidon_desc, elems: *const u64, count: u64, digest_out: *mut u64) -> i32;
        pub fn b2z_prime_search(x: *const u64, j_first: u64, j_last: u64, num_bits: u32, k_bases: u32, threads: u32,
                                out: *mut b2z_prime_check, found: *mut i32) -> i32;
        pub fn b2z_modpow_witnesses(base: u64, modulus: u64, exponent: u64, num_bits: u32, mod_vals: *mut u64,
                                    mod_pow_vals: *mut u64, bits: *mut u8, result: *mut u64) -> i32;
    }
    #[repr(C)]
    pub struct b2z_prime_check {
        pub j: u64, pub digest: [u8; 32], pub is_prime: i32, pub quotient: [u64; 4], pub remainder: u64, pub a: [u64; 4],
    }
    #[repr(C)]
    pub struct b2z_poseidon_desc {
        pub full_rounds: u32, pub partial_rounds: u32, pub alpha: u64, pub width: u32, pub rate: u32, pub capacity: u32,
        pub ark: *const u64, pub mds: *const u64,
    }
}
use sys::*;

// ---------------------------------------------------------------------------------------------- packing
pub fn pack_fr(v: &[Fr]) -> Vec<u64> { v.iter().flat_map(|x| x.0 .0).collect() }               // Montgomery limbs
pub fn pack_bigint(v: &[BigInt<4>]) -> Vec<u64> { v.iter().flat_map(|x| x.0).collect() }       // canonical limbs
pub fn pack_g1(v: &[G1Affine]) -> (Vec<u64>, Vec<u8>) {
    let mut limbs = Vec::with_capacity(v.len() * 12);
    let mut inf = vec![0u8; (v.len() + 7) / 8];
    for (i, p) in v.iter().enumerate() {
        if p.infinity { inf[i >> 3] |= 1 << (i & 7); limbs.extend([0u64; 12]); }
        else { limbs.extend(p.x.0 .0); limbs.extend(p.y.0 .0); }
    }
    (limbs, inf)
}
pub fn pack_g2(v: &[G2Affine]) -> (Vec<u64>, Vec<u8>) {                                        // x.c0, x.c1, y.c0, y.c1
    let mut limbs = Vec::with_capacity(v.len() * 24);
    let mut inf = vec![0u8; (v.len() + 7) / 8];
    for (i, p) in v.iter().enumerate() {
        if p.infinity { inf[i >> 3] |= 1 << (i & 7); limbs.extend([0u64; 24]); }
        else { for c in [&p.x.c0, &p.x.c1, &p.y.c0, &p.y.c1] { limbs.extend(c.0 .0); } }
    }
    (limbs, inf)
}
/// `ConstraintMatrices` row lists -> CSR (row_ptr, cols, Montgomery coefficient limbs) for `b2z_r1cs_upload`.
pub fn to_csr(rows: &[Vec<(Fr, usize)>]) -> (Vec<u64>, Vec<u32>, Vec<u64>) {
    let (mut rp, mut cols, mut cf) = (vec![0u64], Vec::new(), Vec::new());
    for row in rows {
        for (c, j) in row { cols.push(*j as u32); cf.extend(c.0 .0); }
        rp.push(cols.len() as u64);
    }
    (rp, cols, cf)
}
fn unpack_fr(limbs: &[u64]) -> Vec<Fr> {
    limbs.chunks_exact(4).map(|c| ark_ff::Fp(BigInt([c[0], c[1], c[2], c[3]]), core::marker::PhantomData)).collect()
}

fn status(ctx: *const b2z_ctx, st: i32) -> Result<(), SynthesisError> {
    match st {
        B2Z_OK => Ok(()),
        B2Z_ESIZE => Err(SynthesisError::PolynomialDegreeTooLarge),
        _ => {
            if !ctx.is_null() {
                eprintln!("libb200zk: {:?}", unsafe { CStr::from_ptr(b2z_last_error(ctx)) });
            }
            Err(SynthesisError::Unsatisfiable)
        }
    }
}

// ---------------------------------------------------------------------------------------------- context, key
/// One per actix worker thread (/root/reference/src/main.rs:37): calls on a context serialise, and every uploaded
/// key / matrix handle belongs to the context it was uploaded through.
pub struct Context { raw: *mut b2z_ctx }
unsafe impl Send for Context {}
impl Context {
    pub fn new(device: i32) -> Result<Self, SynthesisError> {
        let mut raw = ptr::null_mut();
        status(ptr::null(), unsafe { b2z_ctx_create(device, &mut raw) })?;
        Ok(Self { raw })
    }
}
impl Drop for Context { fn drop(&mut self) { unsafe { b2z_ctx_destroy(self.raw) } } }

/// Device copy of a `ProvingKey<Bls12_381>` (uploaded once per circuit; the reference re-runs setup per request,
/// matrix_proof.rs:129, so the natural place is right after it, cached by circuit shape).
pub struct DeviceKey<'c> { ctx: &'c Context, raw: *mut b2z_pk }
impl<'c> DeviceKey<'c> {
    pub fn upload(ctx: &'c Context, pk: &ProvingKey<Bls12_381>, num_constraints: usize) -> Result<Self, SynthesisError> {
        let (a, a_inf) = pack_g1(&pk.a_query);
        let (b1, b1_inf) = pack_g1(&pk.b_g1_query);
        let (b2, b2_inf) = pack_g2(&pk.b_g2_query);
        let (h, h_inf) = pack_g1(&pk.h_query);
        let (l, l_inf) = pack_g1(&pk.l_query);
        let one = |p: &G1Affine| pack_g1(std::slice::from_ref(p)).0;
        let one2 = |p: &G2Affine| pack_g2(std::slice::from_ref(p)).0;
        let (al, be, de) = (one(&pk.vk.alpha_g1), one(&pk.beta_g1), one(&pk.delta_g1));
        let (be2, de2) = (one2(&pk.vk.beta_g2), one2(&pk.vk.delta_g2));
        let num_instance = pk.vk.gamma_abc_g1.len() as u64;
        let desc = b2z_pk_desc {
            num_variables: pk.a_query.len() as u64, num_instance,
            log_domain: (num_constraints as u64 + num_instance).next_power_of_two().trailing_zeros(),
            a_query: a.as_ptr(), a_inf: a_inf.as_ptr(), b_g1_query: b1.as_ptr(), b_g1_inf: b1_inf.as_ptr(),
            b_g2_query: b2.as_ptr(), b_g2_inf: b2_inf.as_ptr(), h_query: h.as_ptr(), h_inf: h_inf.as_ptr(),
            l_query: l.as_ptr(), l_inf: l_inf.as_ptr(),
            alpha_g1: al.as_ptr(), beta_g1: be.as_ptr(), delta_g1: de.as_ptr(), beta_g2: be2.as_ptr(), delta_g2: de2.as_ptr(),
        };
        let mut raw = ptr::null_mut();
        status(ctx.raw, unsafe { b2z_pk_upload(ctx.raw, &desc, &mut raw) })?;
        Ok(Self { ctx, raw })
    }
}
impl<'c> DeviceKey<'c> {
    /// `Groth16::<Bls12_381>::setup(circuit, rng)` after synthesis, with the key made on the GPU (b2z_groth16_setup):
    /// the draws are arkworks' own, in its order (alpha, beta, gamma, delta, g1, g2, tau), so the key and the
    /// verifying key equal what `Groth16::setup` returns for the same rng.  `m`: the circuit's matrices on `ctx`.
    pub fn setup<R: RngCore>(ctx: &'c Context, m: &DeviceMatrices<'c>, num_constraints: usize, num_instance: usize,
                             rng: &mut R) -> Result<(Self, VerifyingKey<Bls12_381>), SynthesisError> {
        Self::setup_shard(ctx, m, num_constraints, num_instance, 0, 1, rng)
    }
    /// The same setup straight into shard `rank` of `world` of the key (b2z_groth16_setup_shard), the shard that
    /// b2z_pk_upload_shard makes of the whole key: each GPU of a multi-GPU box calls this with an rng seeded alike, so
    /// every rank makes the same draws, and gets its own key shard for the tile-sharded prover and the whole
    /// verifying key.  world == 1: the whole key, as `setup`.
    pub fn setup_shard<R: RngCore>(ctx: &'c Context, m: &DeviceMatrices<'c>, num_constraints: usize,
                                   num_instance: usize, rank: u32, world: u32, rng: &mut R)
                                   -> Result<(Self, VerifyingKey<Bls12_381>), SynthesisError> {
        let domain = ark_poly::Radix2EvaluationDomain::<Fr>::new(num_constraints + num_instance)
            .ok_or(SynthesisError::PolynomialDegreeTooLarge)?;
        let (alpha, beta, gamma, delta) = (Fr::rand(rng), Fr::rand(rng), Fr::rand(rng), Fr::rand(rng));
        let g1 = G1Projective::rand(rng);
        let g2 = G2Projective::rand(rng);
        let tau = loop {
            let t = Fr::rand(rng);
            if !domain.evaluate_vanishing_polynomial(t).is_zero() { break t; }
        };
        let (g1a, g2a): (G1Affine, G2Affine) = (g1.into(), g2.into());
        let (g1l, g2l) = (pack_g1(&[g1a]).0, pack_g2(&[g2a]).0);
        let els = pack_fr(&[alpha, beta, gamma, delta, tau]);
        let desc = b2z_setup_desc {
            alpha: els[0..].as_ptr(), beta: els[4..].as_ptr(), gamma: els[8..].as_ptr(), delta: els[12..].as_ptr(),
            tau: els[16..].as_ptr(), g1_generator: g1l.as_ptr(), g2_generator: g2l.as_ptr(),
        };
        let mut gabc = vec![0u64; num_instance * 12];
        let mut gabc_inf = vec![0u8; (num_instance + 7) / 8];
        let mut vk = b2z_vk_out {
            alpha_g1: [0; 12], beta_g2: [0; 24], gamma_g2: [0; 24], delta_g2: [0; 24],
            gamma_abc_g1: gabc.as_mut_ptr(), gamma_abc_inf: gabc_inf.as_mut_ptr(),
        };
        let mut raw = ptr::null_mut();
        status(ctx.raw, unsafe { b2z_groth16_setup_shard(ctx.raw, m.raw, &desc, rank, world, &mut raw, &mut vk) })?;
        let g1_of = |l: &[u64], inf: bool| -> G1Affine {
            if inf { return G1Affine::identity(); }
            G1Affine::new_unchecked(unpack_fq(&l[0..6]), unpack_fq(&l[6..12]))
        };
        let g2_of = |l: &[u64]| -> G2Affine {
            let f2 = |a: &[u64]| ark_bls12_381::Fq2::new(unpack_fq(&a[0..6]), unpack_fq(&a[6..12]));
            G2Affine::new_unchecked(f2(&l[0..12]), f2(&l[12..24]))
        };
        let vk = VerifyingKey {
            alpha_g1: g1_of(&vk.alpha_g1, false), beta_g2: g2_of(&vk.beta_g2), gamma_g2: g2_of(&vk.gamma_g2),
            delta_g2: g2_of(&vk.delta_g2),
            gamma_abc_g1: (0..num_instance).map(|i| g1_of(&gabc[i * 12..i * 12 + 12], (gabc_inf[i >> 3] >> (i & 7)) & 1 == 1))
                .collect(),
        };
        Ok((Self { ctx, raw }, vk))
    }
}
fn unpack_fq(l: &[u64]) -> ark_bls12_381::Fq {
    ark_ff::Fp(BigInt([l[0], l[1], l[2], l[3], l[4], l[5]]), core::marker::PhantomData)
}
impl Drop for DeviceKey<'_> { fn drop(&mut self) { unsafe { b2z_pk_free(self.ctx.raw, self.raw) } } }

/// Device copy of the circuit's `ConstraintMatrices` (CSR), uploaded once per circuit shape.
pub struct DeviceMatrices<'c> { ctx: &'c Context, raw: *mut b2z_r1cs }
impl<'c> DeviceMatrices<'c> {
    pub fn upload(ctx: &'c Context, m: &ConstraintMatrices<Fr>) -> Result<Self, SynthesisError> {
        let (a, b, c) = (to_csr(&m.a), to_csr(&m.b), to_csr(&m.c));
        let mut raw = ptr::null_mut();
        status(ctx.raw, unsafe {
            b2z_r1cs_upload(ctx.raw, m.num_constraints as u64, m.num_instance_variables as u64,
                            (m.num_instance_variables + m.num_witness_variables) as u64,
                            a.0.as_ptr(), a.1.as_ptr(), a.2.as_ptr(), b.0.as_ptr(), b.1.as_ptr(), b.2.as_ptr(),
                            c.0.as_ptr(), c.1.as_ptr(), c.2.as_ptr(), &mut raw)
        })?;
        Ok(Self { ctx, raw })
    }
}
impl Drop for DeviceMatrices<'_> { fn drop(&mut self) { unsafe { b2z_r1cs_free(self.ctx.raw, self.raw) } } }

// ---------------------------------------------------------------------------------------------- Groth16::prove
pub struct B200Groth16;
impl B200Groth16 {
    /// `ark_groth16::Groth16::<Bls12_381>::prove(&pk, circuit, rng)` = `create_random_proof_with_reduction`:
    /// draws r then s exactly as arkworks does, synthesises in Rust, and leaves the row evaluation, the witness map,
    /// the five MSMs and the serialization to the GPU library.  `dev_m`: the circuit's matrices on the device
    /// (None = evaluate the rows here and send a, b, c).
    pub fn prove<C: ConstraintSynthesizer<Fr>, R: RngCore>(ctx: &Context, dev_pk: &DeviceKey, dev_m: Option<&DeviceMatrices>,
                                                           circuit: C, rng: &mut R) -> Result<Proof<Bls12_381>, SynthesisError> {
        let r = Fr::rand(rng);
        let s = Fr::rand(rng);
        let cs = ConstraintSystem::new_ref();
        cs.set_optimization_goal(OptimizationGoal::Constraints);
        circuit.generate_constraints(cs.clone())?;
        cs.finalize();
        let z = full_assignment(&cs);
        let mut bytes = [0u8; 192];
        let st = match dev_m {
            Some(m) => unsafe {
                b2z_groth16_prove_r1cs(ctx.raw, dev_pk.raw, m.raw, pack_fr(&z).as_ptr(), r.0 .0.as_ptr(), s.0 .0.as_ptr(),
                                       bytes.as_mut_ptr())
            },
            None => {
                let m = cs.to_matrices().ok_or(SynthesisError::AssignmentMissing)?;
                let (a, b, c) = constraint_evaluations(&m, &z)?;
                unsafe {
                    b2z_groth16_prove(ctx.raw, dev_pk.raw, pack_fr(&a).as_ptr(), pack_fr(&b).as_ptr(), pack_fr(&c).as_ptr(),
                                      pack_fr(&z).as_ptr(), r.0 .0.as_ptr(), s.0 .0.as_ptr(), bytes.as_mut_ptr())
                }
            }
        };
        status(ctx.raw, st)?;
        Proof::deserialize_compressed(&bytes[..]).map_err(|_| SynthesisError::Unsatisfiable)
    }
}

fn full_assignment(cs: &ConstraintSystemRef<Fr>) -> Vec<Fr> {
    let p = cs.borrow().unwrap();
    [&p.instance_assignment[..], &p.witness_assignment[..]].concat()
}

/// The a, b, c vectors `witness_map_from_matrices` builds before its FFTs.
pub fn constraint_evaluations(m: &ConstraintMatrices<Fr>, z: &[Fr]) -> Result<(Vec<Fr>, Vec<Fr>, Vec<Fr>), SynthesisError> {
    let n = (m.num_constraints + m.num_instance_variables).next_power_of_two();
    if n.trailing_zeros() > 32 { return Err(SynthesisError::PolynomialDegreeTooLarge); }
    let dot = |row: &[(Fr, usize)]| row.iter().fold(Fr::zero(), |acc, (c, j)| acc + *c * z[*j]);
    let (mut a, mut b, mut c) = (vec![Fr::zero(); n], vec![Fr::zero(); n], vec![Fr::zero(); n]);
    for i in 0..m.num_constraints { a[i] = dot(&m.a[i]); b[i] = dot(&m.b[i]); c[i] = dot(&m.c[i]); }
    a[m.num_constraints..m.num_constraints + m.num_instance_variables].clone_from_slice(&z[..m.num_instance_variables]);
    Ok((a, b, c))
}

// ---------------------------------------------------------------------------------------------- R1CSToQAP
/// `Groth16::<Bls12_381, B200Reduction>` keeps ark-groth16's own prover and swaps only the witness map.
/// The context comes from a thread-local because the trait has no `self`.
pub struct B200Reduction;
thread_local! { pub static CTX: Context = Context::new(0).expect("no CUDA device: libb200zk has no CPU fallback"); }
impl R1CSToQAP for B200Reduction {
    fn instance_map_with_evaluation<F: PrimeField, D: EvaluationDomain<F>>(cs: ConstraintSystemRef<F>, t: &F)
        -> Result<(Vec<F>, Vec<F>, Vec<F>, F, usize, usize), SynthesisError> {
        ark_groth16::r1cs_to_qap::LibsnarkReduction::instance_map_with_evaluation::<F, D>(cs, t)     // setup side: unchanged
    }
    fn witness_map_from_matrices<F: PrimeField, D: EvaluationDomain<F>>(matrices: &ConstraintMatrices<F>, num_inputs: usize,
                                                                         num_constraints: usize, full_assignment: &[F])
        -> Result<Vec<F>, SynthesisError> {
        // Only Fr of BLS12-381 is accelerated; the limbs are copied, so the cast is by value, not by transmute.
        assert_eq!(F::MODULUS_BIT_SIZE, 255, "B200Reduction is specialised to the BLS12-381 scalar field");
        let limbs = |x: &F| -> [u64; 4] { let b = x.into_bigint(); let v = b.as_ref(); [v[0], v[1], v[2], v[3]] };
        let to_fr = |x: &F| Fr::from_bigint(BigInt(limbs(x))).unwrap();
        let z: Vec<Fr> = full_assignment.iter().map(to_fr).collect();
        let conv = |rows: &Vec<Vec<(F, usize)>>| -> Vec<Vec<(Fr, usize)>> {
            rows.iter().map(|r| r.iter().map(|(c, j)| (to_fr(c), *j)).collect()).collect()
        };
        let m = ConstraintMatrices::<Fr> {
            num_instance_variables: num_inputs, num_witness_variables: matrices.num_witness_variables,
            num_constraints, a_num_non_zero: matrices.a_num_non_zero, b_num_non_zero: matrices.b_num_non_zero,
            c_num_non_zero: matrices.c_num_non_zero, a: conv(&matrices.a), b: conv(&matrices.b), c: conv(&matrices.c),
        };
        let (a, b, c) = constraint_evaluations(&m, &z)?;
        let n = a.len();
        let mut h = vec![0u64; 4 * n];
        CTX.with(|ctx| status(ctx.raw, unsafe {
            b2z_witness_map(ctx.raw, pack_fr(&a).as_ptr(), pack_fr(&b).as_ptr(), pack_fr(&c).as_ptr(), n.trailing_zeros(),
                            h.as_mut_ptr())
        }))?;
        Ok(unpack_fr(&h).iter().map(|x| F::from_bigint(F::BigInt::try_from(num_bigint(x)).ok().unwrap()).unwrap()).collect())
    }
    fn h_query_scalars<F: PrimeField, D: EvaluationDomain<F>>(max_power: usize, t: F, zt: F, delta_inverse: F)
        -> Result<Vec<F>, SynthesisError> {
        ark_groth16::r1cs_to_qap::LibsnarkReduction::h_query_scalars::<F, D>(max_power, t, zt, delta_inverse)
    }
}
fn num_bigint(x: &Fr) -> ark_std::vec::Vec<u8> { use ark_ff::BigInteger; x.into_bigint().to_bytes_le() }

// ---------------------------------------------------------------------------------------------- MSM, NTT
/// `<G1Projective as VariableBaseMSM>::msm_bigint(bases, scalars)`.
pub fn msm_bigint_g1(ctx: &Context, bases: &[G1Affine], scalars: &[BigInt<4>]) -> Result<G1Projective, SynthesisError> {
    let n = bases.len().min(scalars.len());
    let (b, inf) = pack_g1(&bases[..n]);
    let mut out = [0u64; 18];
    status(ctx.raw, unsafe { b2z_msm_g1(ctx.raw, b.as_ptr(), inf.as_ptr(), pack_bigint(&scalars[..n]).as_ptr(), n as u64, out.as_mut_ptr()) })?;
    let f = |o: usize| ark_bls12_381::Fq::new_unchecked(BigInt([out[o], out[o + 1], out[o + 2], out[o + 3], out[o + 4], out[o + 5]]));
    Ok(G1Projective::new_unchecked(f(0), f(6), f(12)))
}
/// `<G2Projective as VariableBaseMSM>::msm_bigint(bases, scalars)`.
pub fn msm_bigint_g2(ctx: &Context, bases: &[G2Affine], scalars: &[BigInt<4>]) -> Result<G2Projective, SynthesisError> {
    let n = bases.len().min(scalars.len());
    let (b, inf) = pack_g2(&bases[..n]);
    let mut out = [0u64; 36];
    status(ctx.raw, unsafe { b2z_msm_g2(ctx.raw, b.as_ptr(), inf.as_ptr(), pack_bigint(&scalars[..n]).as_ptr(), n as u64, out.as_mut_ptr()) })?;
    let f = |o: usize| ark_bls12_381::Fq::new_unchecked(BigInt([out[o], out[o + 1], out[o + 2], out[o + 3], out[o + 4], out[o + 5]]));
    let f2 = |o: usize| ark_bls12_381::Fq2::new(f(o), f(o + 6));
    Ok(G2Projective::new_unchecked(f2(0), f2(12), f2(24)))
}
/// `domain.fft_in_place` / `ifft_in_place` (coset: `domain.get_coset(g)`), natural order in and out.
pub fn ntt_in_place(ctx: &Context, data: &mut [Fr], inverse: bool, coset: Option<Fr>) -> Result<(), SynthesisError> {
    assert!(data.len().is_power_of_two());
    let mut limbs = pack_fr(data);
    let g = coset.map(|g| g.0 .0);
    status(ctx.raw, unsafe {
        b2z_ntt_fr(ctx.raw, limbs.as_mut_ptr(), data.len().trailing_zeros(), inverse as i32,
                   g.as_ref().map_or(ptr::null(), |x| x.as_ptr()))
    })?;
    data.clone_from_slice(&unpack_fr(&limbs));
    Ok(())
}

// ---------------------------------------------------------------------------------------------- verifier (host only)
/// `prepare_verifying_key(&vk)` + `serialize_compressed`: the bytes `encode_pvk` base64-encodes (io.rs:62-68).
/// `hasher()` of the reference (matrix_proof_of_work/hasher.rs:17-27) on the host cores of the GPU box, with the
/// caller's own `PoseidonConfig` (hashing_utils.rs: `poseidon_parameters_for_test`): absorb everything, squeeze one.
pub fn poseidon_hash(cfg: &ark_crypto_primitives::sponge::poseidon::PoseidonConfig<Fr>, elems: &[Fr]) -> Result<Fr, SynthesisError> {
    let ark: Vec<u64> = cfg.ark.iter().flat_map(|row| row.iter().flat_map(|x| x.0 .0)).collect();
    let mds: Vec<u64> = cfg.mds.iter().flat_map(|row| row.iter().flat_map(|x| x.0 .0)).collect();
    let d = b2z_poseidon_desc {
        full_rounds: cfg.full_rounds as u32, partial_rounds: cfg.partial_rounds as u32, alpha: cfg.alpha,
        width: (cfg.rate + cfg.capacity) as u32, rate: cfg.rate as u32, capacity: cfg.capacity as u32,
        ark: ark.as_ptr(), mds: mds.as_ptr(),
    };
    let mut out = [0u64; 4];
    let st = unsafe { b2z_poseidon_hash(&d, pack_fr(elems).as_ptr(), elems.len() as u64, out.as_mut_ptr()) };
    if st != B2Z_OK { return Err(SynthesisError::AssignmentMissing); }
    Ok(ark_ff::Fp(BigInt(out), core::marker::PhantomData))
}

pub fn prepared_vk_bytes(vk: &VerifyingKey<Bls12_381>) -> Result<Vec<u8>, SynthesisError> {
    let one = |p: &G1Affine| pack_g1(std::slice::from_ref(p)).0;
    let one2 = |p: &G2Affine| pack_g2(std::slice::from_ref(p)).0;
    let (al, be, ga, de) = (one(&vk.alpha_g1), one2(&vk.beta_g2), one2(&vk.gamma_g2), one2(&vk.delta_g2));
    let (abc, abc_inf) = pack_g1(&vk.gamma_abc_g1);
    let desc = b2z_vk_desc { num_instance: vk.gamma_abc_g1.len() as u64, alpha_g1: al.as_ptr(), beta_g2: be.as_ptr(),
                             gamma_g2: ga.as_ptr(), delta_g2: de.as_ptr(), gamma_abc_g1: abc.as_ptr(), gamma_abc_inf: abc_inf.as_ptr() };
    let mut len = 0u64;
    status(ptr::null(), unsafe { b2z_groth16_prepare_verifying_key(&desc, ptr::null_mut(), 0, &mut len) })?;
    let mut out = vec![0u8; len as usize];
    status(ptr::null(), unsafe { b2z_groth16_prepare_verifying_key(&desc, out.as_mut_ptr(), len, &mut len) })?;
    Ok(out)
}
/// `Groth16::<Bls12_381>::verify_with_processed_vk(&pvk, inputs, &proof)` on the wire bytes (matrix_proof.rs:199-206).
pub fn verify_with_processed_vk(pvk: &[u8], public_inputs: &[Fr], proof: &[u8; 192]) -> Result<bool, SynthesisError> {
    let mut valid = 0i32;
    let st = unsafe {
        b2z_groth16_verify_with_processed_vk(pvk.as_ptr(), pvk.len() as u64, pack_fr(public_inputs).as_ptr(),
                                             public_inputs.len() as u64, proof.as_ptr(), &mut valid)
    };
    if st != B2Z_OK { return Err(SynthesisError::MalformedVerifyingKey); }
    Ok(valid == 1)
}

/// `verify_with_processed_vk` for many proofs against one pvk on ctx's GPU (b2z_groth16_verify_batch): one verdict
/// per proof, `None` where the single-proof call would return an error (malformed encoding, point outside the
/// subgroup).  Every proof takes the same number of inputs.  Err for what fails the whole call: malformed pvk, a
/// wrong input count, more than 1024 inputs.
pub fn verify_batch_with_processed_vk(ctx: &Context, pvk: &[u8], inputs: &[Vec<Fr>], proofs: &[[u8; 192]])
                                      -> Result<Vec<Option<bool>>, SynthesisError> {
    if inputs.len() != proofs.len() { return Err(SynthesisError::MalformedVerifyingKey); }
    if proofs.is_empty() { return Ok(Vec::new()); }
    let n = inputs[0].len();
    if inputs.iter().any(|x| x.len() != n) { return Err(SynthesisError::MalformedVerifyingKey); }
    let x: Vec<u64> = inputs.iter().flat_map(|v| pack_fr(v)).collect();
    let bytes: Vec<u8> = proofs.iter().flat_map(|p| p.iter().copied()).collect();
    let mut results = vec![0i32; proofs.len()];
    let st = unsafe {
        b2z_groth16_verify_batch(ctx.raw, pvk.as_ptr(), pvk.len() as u64, if n > 0 { x.as_ptr() } else { ptr::null() },
                                 n as u64, bytes.as_ptr(), proofs.len() as u64, results.as_mut_ptr())
    };
    match st {
        B2Z_OK => Ok(results.iter().map(|&r| if r < 0 { None } else { Some(r == 1) }).collect()),
        B2Z_EINVAL | B2Z_ESIZE => Err(SynthesisError::MalformedVerifyingKey),
        _ => status(ctx.raw, st).map(|_| Vec::new()),
    }
}

#[allow(dead_code)]
fn _type_checks(p: G1Affine) -> bool { p.is_zero() && Fr::zero().inverse().is_none() }
