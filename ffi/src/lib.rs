//! h2v-sys -- Rust binding of `include/h2v.h` plus safe wrappers with the exact halo2-axiom signatures the
//! reference reaches through `src/scaffold/mod.rs:273` (create_pk) and `:296` (gen_snark_shplonk):
//! `best_multiexp`, `best_fft`, `ParamsKZG::{commit, commit_lagrange}` and
//! `EvaluationDomain::{lagrange_to_coeff, coeff_to_extended, extended_to_coeff, divide_by_vanishing_poly}`.
//!
//! SOURCE ONLY: not compiled in this repository's image (no cargo).  `Fr`, `G1Affine`, `G1` of halo2curves
//! are `#[repr(C)]`-compatible `[u64; 4]` Montgomery limbs (identity affine = (0,0)), which is exactly the
//! ABI's layout, so slices are passed by pointer with no conversion.
//!
//! Error behaviour: upstream panics (`assert_eq!(a.len(), 1 << log_n)`, length mismatch) stay panics;
//! any CUDA failure is also a panic -- there is no CPU fallback.
use halo2curves::bn256::{Fr, G1Affine, G1};
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct H2vSrs(c_void);
#[repr(C)]
pub struct H2vDomain(c_void);

#[repr(C)] pub struct H2vPk { _private: [u8; 0] }
#[repr(C)] pub struct H2vBuilder { _private: [u8; 0] }
#[repr(C)] pub struct H2vWitnessProgram { _private: [u8; 0] }
/// `h2v_circuit_t`: the constraint-system description `h2v_pk_load` takes (include/h2v.h)
#[repr(C)]
pub struct H2vCircuit {
    pub k: u32, pub degree: u32, pub blinding_factors: u32,
    pub n_advice: u32, pub n_fixed: u32, pub n_instance: u32,
    pub n_gates: u32, pub gate_advice: *const u32, pub gate_selector: *const u32,
    pub n_lookups: u32, pub lookup_input: *const u32, pub lookup_table: *const u32,
    pub n_perm: u32, pub perm_kind: *const u8, pub perm_index: *const u32,
    pub n_advice_queries: u32, pub advice_query_col: *const u32, pub advice_query_rot: *const i32,
    pub n_fixed_queries: u32, pub fixed_query_col: *const u32, pub fixed_query_rot: *const i32,
}
/// `h2v_mock_failure_t`: one failed constraint of `h2v_mock_prover` (kind = H2V_MOCK_*)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct H2vMockFailure { pub kind: u32, pub column: u32, pub row: u32, pub other_column: u32, pub other_row: u32 }
pub const H2V_MOCK_GATE: u32 = 1;
pub const H2V_MOCK_GATE_UNUSABLE: u32 = 2;
pub const H2V_MOCK_LOOKUP: u32 = 3;
pub const H2V_MOCK_SIGMA_NOT_DELTA_OMEGA: u32 = 4;
pub const H2V_MOCK_SIGMA_NOT_PERMUTATION: u32 = 5;
pub const H2V_MOCK_COPY_UNUSABLE: u32 = 6;
pub const H2V_MOCK_COPY: u32 = 7;
pub const H2V_BASIS_MONOMIAL: c_int = 0;
pub const H2V_BASIS_LAGRANGE: c_int = 1;
pub const H2V_OP_LAGRANGE_TO_COEFF: c_int = 0;
pub const H2V_OP_COEFF_TO_LAGRANGE: c_int = 1;
pub const H2V_OP_COEFF_TO_EXTENDED: c_int = 2;
pub const H2V_OP_EXTENDED_TO_COEFF: c_int = 3;
pub const H2V_OP_DIVIDE_BY_VANISHING: c_int = 4;

extern "C" {
    pub fn h2v_init(devices: *const c_int, n_dev: c_int) -> c_int;
    pub fn h2v_device_count() -> c_int;
    pub fn h2v_last_error() -> *const c_char;
    pub fn h2v_host_register(ptr: *mut c_void, bytes: usize) -> c_int;
    pub fn h2v_host_unregister(ptr: *mut c_void) -> c_int;
    pub fn h2v_srs_load(k: u32, g: *const u64, g_lagrange: *const u64, out: *mut *mut H2vSrs) -> c_int;
    pub fn h2v_srs_free(srs: *mut H2vSrs);
    pub fn h2v_commit(srs: *mut H2vSrs, basis: c_int, poly: *const u64, len: usize, out_affine: *mut u64) -> c_int;
    pub fn h2v_commit_batch(srs: *mut H2vSrs, basis: c_int, polys: *const *const u64, n_polys: usize, len: usize,
                            out_affine: *mut u64) -> c_int;
    pub fn h2v_best_multiexp(coeffs: *const u64, bases: *const u64, n: usize, out_jacobian: *mut u64) -> c_int;
    pub fn h2v_best_fft(a: *mut u64, omega: *const u64, log_n: u32) -> c_int;
    pub fn h2v_domain_new(j: u32, k: u32, out: *mut *mut H2vDomain) -> c_int;
    pub fn h2v_domain_free(dom: *mut H2vDomain);
    pub fn h2v_domain_extended_k(dom: *mut H2vDomain) -> u32;
    pub fn h2v_lagrange_to_coeff(dom: *mut H2vDomain, a: *mut u64) -> c_int;
    pub fn h2v_coeff_to_lagrange(dom: *mut H2vDomain, a: *mut u64) -> c_int;
    pub fn h2v_coeff_to_extended(dom: *mut H2vDomain, inp: *const u64, out: *mut u64) -> c_int;
    pub fn h2v_extended_to_coeff(dom: *mut H2vDomain, inp: *const u64, out: *mut u64) -> c_int;
    pub fn h2v_divide_by_vanishing_poly(dom: *mut H2vDomain, a: *mut u64) -> c_int;
    pub fn h2v_domain_transform_batch(dom: *mut H2vDomain, op: c_int, inp: *const *const u64, out: *const *mut u64,
                                      n_cols: usize) -> c_int;
    pub fn h2v_srs_setup(k: u32, s_mont: *const u64, g_out: *mut u64, g_lagrange_out: *mut u64) -> c_int;
    // polynomial primitives around the commits (SURVEY.md 8(f) row 2)
    pub fn h2v_eval_polynomial_batch(polys: *const *const u64, n_polys: usize, len: usize, points: *const u64,
                                     n_points: usize, out: *mut u64) -> c_int;
    pub fn h2v_batch_invert(a: *mut u64, n: usize) -> c_int;
    pub fn h2v_grand_product(num: *const u64, den: *const u64, n: usize, out: *mut u64) -> c_int;
    pub fn h2v_kate_division(a: *const u64, n: usize, b: *const u64, out: *mut u64) -> c_int;
    // device-resident columns
    pub fn h2v_dev_alloc(bytes: usize, d_out: *mut *mut c_void) -> c_int;
    pub fn h2v_dev_free(d_ptr: *mut c_void) -> c_int;
    pub fn h2v_dev_upload(d_dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn h2v_dev_download(dst: *mut c_void, d_src: *const c_void, bytes: usize) -> c_int;
    pub fn h2v_commit_batch_resident(srs: *mut H2vSrs, basis: c_int, polys: *const *const u64, n_polys: usize, len: usize, tails: *const u64,
                                     row0: usize, n_rows: usize, d_dst: *mut c_void, dst_stride: usize, out_affine: *mut u64) -> c_int;
    pub fn h2v_commit_batch_dev(srs: *mut H2vSrs, basis: c_int, d_polys: *const c_void, col_stride: usize, n_polys: usize,
                                len: usize, d_out_affine: *mut c_void) -> c_int;
    pub fn h2v_domain_transform_dev(dom: *mut H2vDomain, op: c_int, d_in: *const c_void, in_stride: usize,
                                    d_out: *mut c_void, out_stride: usize, n_cols: usize) -> c_int;
    pub fn h2v_permute_expression_pair(input: *const u64, table: *const u64, usable_rows: usize, permuted_input: *mut u64,
                                       permuted_table: *mut u64) -> c_int;
    pub fn h2v_g1_sum(affine_pts: *const u64, n: usize, out_affine: *mut u64) -> c_int;
    // poly/domain.rs helpers (SURVEY.md 8(a) row a12)
    pub fn h2v_domain_rotate_omega(dom: *mut H2vDomain, value: *const u64, rotation: i32, out: *mut u64) -> c_int;
    pub fn h2v_domain_rotate_extended(dom: *mut H2vDomain, inp: *const u64, rotation: i32, out: *mut u64) -> c_int;
    pub fn h2v_domain_l_i_range(dom: *mut H2vDomain, x: *const u64, xn: *const u64, rot_lo: i32, rot_hi: i32, out: *mut u64) -> c_int;
    pub fn h2v_domain_fill(dom: *mut H2vDomain, basis: c_int, scalar: *const u64, out: *mut u64) -> c_int;
    // gen_srs (scaffold mod.rs:260): seeded setup, .srs file
    pub fn h2v_srs_gen(k: u32, seed: *const u8, g_out: *mut u64, g_lagrange_out: *mut u64, g2_out: *mut u64, s_g2_out: *mut u64) -> c_int;
    pub fn h2v_srs_write_file(path: *const c_char, k: u32, g: *const u64, g_lagrange: *const u64, g2: *const u64, s_g2: *const u64) -> c_int;
    pub fn h2v_srs_read_file(path: *const c_char, k_out: *mut u32, g: *mut u64, g_lagrange: *mut u64, cap_points: usize, g2: *mut u64,
                             s_g2: *mut u64) -> c_int;
    // create_proof (plonk/prover.rs) on the device, transcript (SURVEY.md 8(f) rows 2-3)
    pub fn h2v_pk_load(srs: *mut H2vSrs, cs: *const H2vCircuit, fixed: *const *const u64, sigma: *const *const u64, vk_repr: *const u64,
                       out: *mut *mut H2vPk) -> c_int;
    pub fn h2v_pk_free(pk: *mut H2vPk);
    pub fn h2v_proof_size(pk: *mut H2vPk) -> usize;
    pub fn h2v_create_proof(pk: *mut H2vPk, advice: *const *const u64, instances: *const *const u64, instance_len: *const u32,
                            rng_seed: *const u8, proof_out: *mut u8, proof_cap: usize, proof_len: *mut usize) -> c_int;
    pub fn h2v_create_proofs(pk: *mut H2vPk, n_proofs: usize, advice: *const *const *const u64, instances: *const *const *const u64,
                             instance_len: *const *const u32, rng_seeds: *const u8, proofs_out: *mut u8, proof_stride: usize) -> c_int;
    pub fn h2v_mock_prover(cs: *const H2vCircuit, fixed: *const *const u64, sigma: *const *const u64, advice: *const *const u64,
                           instances: *const *const u64, instance_len: *const u32, failures_out: *mut H2vMockFailure, cap: usize,
                           n_failures: *mut u64) -> c_int;
    pub fn h2v_pk_mock_prover(pk: *mut H2vPk, n_witnesses: usize, advice: *const *const *const u64, instances: *const *const *const u64,
                              instance_len: *const *const u32, failures_out: *mut H2vMockFailure, cap: usize, n_failures: *mut u64) -> c_int;
    // witness generation on the device for many inputs of one recorded circuit (halo2-base `witness_gen_only`)
    pub fn h2v_builder_new_recording(precision_bits: u32, lookup_bits: u32, out: *mut *mut H2vBuilder) -> c_int;
    pub fn h2v_builder_free(b: *mut H2vBuilder);
    pub fn h2v_witness_program_new(b: *mut H2vBuilder, k: u32, minimum_rows: u32, out: *mut *mut H2vWitnessProgram) -> c_int;
    pub fn h2v_witness_program_free(p: *mut H2vWitnessProgram);
    pub fn h2v_witness_program_info(p: *mut H2vWitnessProgram, out: *mut u64) -> c_int;
    pub fn h2v_witness_program_inputs(p: *mut H2vWitnessProgram, out: *mut u64) -> c_int;
    pub fn h2v_witness_generate(p: *mut H2vWitnessProgram, n_witnesses: usize, n_inputs: usize, inputs: *const u64, advice_out: *mut u64,
                                instances_out: *mut u64) -> c_int;
    pub fn h2v_witness_last_ms(out: *mut f64) -> c_int;
    pub fn h2v_create_proofs_from_inputs(pk: *mut H2vPk, prog: *mut H2vWitnessProgram, n_proofs: usize, n_inputs: usize, inputs: *const u64,
                                         rng_seeds: *const u8, proofs_out: *mut u8, proof_stride: usize, instances_out: *mut u64) -> c_int;
    pub fn h2v_pk_mock_prover_from_inputs(pk: *mut H2vPk, prog: *mut H2vWitnessProgram, n_witnesses: usize, n_inputs: usize, inputs: *const u64,
                                          failures_out: *mut H2vMockFailure, cap: usize, n_failures: *mut u64) -> c_int;
    pub fn h2v_quotient_gates_dev(dom: *mut H2vDomain, d_h: *mut c_void, y: *const u64, n_gates: usize, d_q: *const c_void,
                                  q_stride: usize, d_a: *const c_void, a_stride: usize) -> c_int;
    pub fn h2v_quotient_permutation_dev(dom: *mut H2vDomain, d_h: *mut c_void, y: *const u64, beta: *const u64, gamma: *const u64,
                                        n_cols: usize, chunk_len: usize, d_cols: *const c_void, cols_stride: usize,
                                        d_sigma: *const c_void, sigma_stride: usize, d_z: *const c_void, z_stride: usize,
                                        d_l0: *const c_void, d_l_last: *const c_void, d_l_active: *const c_void,
                                        blinding_factors: u32) -> c_int;
    pub fn h2v_quotient_permutation_range_ptrs_dev(dom: *mut H2vDomain, d_h: *mut c_void, y: *const u64, beta: *const u64, gamma: *const u64,
                                                   n_cols: usize, chunk_len: usize, set_begin: usize, set_end: usize, with_head: c_int,
                                                   d_col_ptrs: *const *const c_void, d_sigma_ptrs: *const *const c_void,
                                                   d_z: *const c_void, z_stride: usize, d_l0: *const c_void, d_l_last: *const c_void,
                                                   d_l_active: *const c_void, blinding_factors: u32) -> c_int;
    pub fn h2v_quotient_lookup_dev(dom: *mut H2vDomain, d_h: *mut c_void, y: *const u64, beta: *const u64, gamma: *const u64,
                                   d_input: *const c_void, d_table: *const c_void, d_perm_input: *const c_void,
                                   d_perm_table: *const c_void, d_z: *const c_void, d_l0: *const c_void, d_l_last: *const c_void,
                                   d_l_active: *const c_void) -> c_int;
}

/// `MockProver::run(k, circuit, instances)` on the device: (the first `max_failures` failures in the order gates, lookups,
/// permutation; their total).  Columns are Lagrange, 2^k values each; no SRS and no key.
pub fn mock_prover(cs: &H2vCircuit, fixed: &[&[Fr]], sigma: &[&[Fr]], advice: &[&[Fr]], instances: &[&[Fr]],
                   max_failures: usize) -> (Vec<H2vMockFailure>, u64) {
    let n = 1usize << cs.k;
    assert!(fixed.len() == cs.n_fixed as usize && sigma.len() == cs.n_perm as usize && advice.len() == cs.n_advice as usize
            && instances.len() == cs.n_instance as usize);
    assert!(fixed.iter().chain(sigma).chain(advice).all(|c| c.len() == n));
    let ptrs = |cols: &[&[Fr]]| -> Vec<*const u64> { cols.iter().map(|c| c.as_ptr() as *const u64).collect() };
    let (f, s, a, i) = (ptrs(fixed), ptrs(sigma), ptrs(advice), ptrs(instances));
    let il: Vec<u32> = instances.iter().map(|c| c.len() as u32).collect();
    let mut out = vec![H2vMockFailure::default(); max_failures];
    let mut total = 0u64;
    ok(unsafe { h2v_mock_prover(cs, f.as_ptr(), s.as_ptr(), a.as_ptr(), i.as_ptr(), il.as_ptr(), out.as_mut_ptr(), max_failures, &mut total) });
    out.truncate((total as usize).min(max_failures));
    (out, total)
}

/// `plonk::lookup::prover::permute_expression_pair` on the usable rows; `Err(())` = `Error::ConstraintSystemFailure`
pub fn permute_expression_pair(input: &[Fr], table: &[Fr]) -> Result<(Vec<Fr>, Vec<Fr>), ()> {
    assert_eq!(input.len(), table.len());
    let (mut a, mut s) = (vec![Fr::zero(); input.len()], vec![Fr::zero(); input.len()]);
    let rc = unsafe {
        h2v_permute_expression_pair(input.as_ptr() as *const u64, table.as_ptr() as *const u64, input.len(),
                                    a.as_mut_ptr() as *mut u64, s.as_mut_ptr() as *mut u64)
    };
    match rc { 0 => Ok((a, s)), -1 => Err(()), _ => { ok(rc); unreachable!() } }
}

/// `halo2_proofs::arithmetic::eval_polynomial`
pub fn eval_polynomial(poly: &[Fr], point: Fr) -> Fr {
    let ptr = [poly.as_ptr() as *const u64];
    let mut out = Fr::zero();
    ok(unsafe { h2v_eval_polynomial_batch(ptr.as_ptr(), 1, poly.len(), &point as *const Fr as *const u64, 1,
                                          &mut out as *mut Fr as *mut u64) });
    out
}
/// `halo2_proofs::arithmetic::kate_division(a, b)`
pub fn kate_division(a: &[Fr], b: Fr) -> Vec<Fr> {
    let mut out = vec![Fr::zero(); a.len().saturating_sub(1)];
    ok(unsafe { h2v_kate_division(a.as_ptr() as *const u64, a.len(), &b as *const Fr as *const u64, out.as_mut_ptr() as *mut u64) });
    out
}
/// `ff::BatchInvert::batch_invert` on a slice
pub fn batch_invert(a: &mut [Fr]) { ok(unsafe { h2v_batch_invert(a.as_mut_ptr() as *mut u64, a.len()) }) }

fn ok(rc: c_int) {
    if rc != 0 {
        let msg = unsafe { CStr::from_ptr(h2v_last_error()) }.to_string_lossy().into_owned();
        panic!("libh2v: {msg}");
    }
}

/// `halo2_proofs::arithmetic::best_multiexp`
pub fn best_multiexp(coeffs: &[Fr], bases: &[G1Affine]) -> G1 {
    assert_eq!(coeffs.len(), bases.len());
    let mut out = G1::default();
    ok(unsafe { h2v_best_multiexp(coeffs.as_ptr() as *const u64, bases.as_ptr() as *const u64, coeffs.len(),
                                  &mut out as *mut G1 as *mut u64) });
    out
}

/// `halo2_proofs::arithmetic::best_fft` for `G = Fr` (the G1 instantiation is only used by `ParamsKZG::setup`)
pub fn best_fft(a: &mut [Fr], omega: Fr, log_n: u32) {
    assert_eq!(a.len(), 1 << log_n);
    ok(unsafe { h2v_best_fft(a.as_mut_ptr() as *mut u64, &omega as *const Fr as *const u64, log_n) });
}

/// Device-resident bases of a `ParamsKZG<Bn256>`; create once next to the params (`gen_srs`, scaffold mod.rs:260).
pub struct DeviceSrs(*mut H2vSrs);
unsafe impl Send for DeviceSrs {}
unsafe impl Sync for DeviceSrs {}
impl DeviceSrs {
    pub fn new(k: u32, g: &[G1Affine], g_lagrange: &[G1Affine]) -> Self {
        assert_eq!(g.len(), 1 << k);
        assert_eq!(g_lagrange.len(), 1 << k);
        let mut h = std::ptr::null_mut();
        ok(unsafe { h2v_srs_load(k, g.as_ptr() as *const u64, g_lagrange.as_ptr() as *const u64, &mut h) });
        DeviceSrs(h)
    }
    fn commit_basis(&self, basis: c_int, poly: &[Fr]) -> G1 {
        let mut aff = G1Affine::default();
        ok(unsafe { h2v_commit(self.0, basis, poly.as_ptr() as *const u64, poly.len(), &mut aff as *mut G1Affine as *mut u64) });
        aff.into()
    }
    /// `ParamsKZG::commit(&self, poly: &Polynomial<Fr, Coeff>, _: Blind<Fr>) -> G1`
    pub fn commit(&self, poly: &[Fr]) -> G1 { self.commit_basis(H2V_BASIS_MONOMIAL, poly) }
    /// `ParamsKZG::commit_lagrange(&self, poly: &Polynomial<Fr, LagrangeCoeff>, _: Blind<Fr>) -> G1`
    pub fn commit_lagrange(&self, poly: &[Fr]) -> G1 { self.commit_basis(H2V_BASIS_LAGRANGE, poly) }
    /// all columns of one prover phase in a single call (preferred: one launch, shared bases)
    pub fn commit_lagrange_batch(&self, polys: &[&[Fr]]) -> Vec<G1Affine> {
        let len = polys.first().map_or(0, |p| p.len());
        assert!(polys.iter().all(|p| p.len() == len));
        let ptrs: Vec<*const u64> = polys.iter().map(|p| p.as_ptr() as *const u64).collect();
        let mut out = vec![G1Affine::default(); polys.len()];
        ok(unsafe { h2v_commit_batch(self.0, H2V_BASIS_LAGRANGE, ptrs.as_ptr(), polys.len(), len, out.as_mut_ptr() as *mut u64) });
        out
    }
}
impl Drop for DeviceSrs {
    fn drop(&mut self) { unsafe { h2v_srs_free(self.0) } }
}

/// Device twiddles/constants of an `EvaluationDomain<Fr>`; create inside `EvaluationDomain::new(j, k)`.
pub struct DeviceDomain { h: *mut H2vDomain, j: u32, k: u32 }
unsafe impl Send for DeviceDomain {}
unsafe impl Sync for DeviceDomain {}
impl DeviceDomain {
    pub fn new(j: u32, k: u32) -> Self {
        let mut h = std::ptr::null_mut();
        ok(unsafe { h2v_domain_new(j, k, &mut h) });
        DeviceDomain { h, j, k }
    }
    pub fn extended_k(&self) -> u32 { unsafe { h2v_domain_extended_k(self.h) } }
    fn n(&self) -> usize { 1usize << self.k }
    fn extended_n(&self) -> usize { 1usize << self.extended_k() }
    /// `EvaluationDomain::lagrange_to_coeff` (values in place); upstream asserts the length, so do we
    pub fn lagrange_to_coeff(&self, a: &mut [Fr]) {
        assert_eq!(a.len(), self.n());
        ok(unsafe { h2v_lagrange_to_coeff(self.h, a.as_mut_ptr() as *mut u64) })
    }
    pub fn coeff_to_lagrange(&self, a: &mut [Fr]) {
        assert_eq!(a.len(), self.n());
        ok(unsafe { h2v_coeff_to_lagrange(self.h, a.as_mut_ptr() as *mut u64) })
    }
    /// `EvaluationDomain::coeff_to_extended`: `a.len() == 2^k`, result `2^extended_k`
    pub fn coeff_to_extended(&self, a: &[Fr]) -> Vec<Fr> {
        assert_eq!(a.len(), self.n());
        let mut out = vec![Fr::zero(); self.extended_n()];
        ok(unsafe { h2v_coeff_to_extended(self.h, a.as_ptr() as *const u64, out.as_mut_ptr() as *mut u64) });
        out
    }
    /// `EvaluationDomain::extended_to_coeff`: `a.len() == 2^extended_k`, result `2^k * (j - 1)` (computed here, not by the caller)
    pub fn extended_to_coeff(&self, a: &[Fr]) -> Vec<Fr> {
        assert_eq!(a.len(), self.extended_n());
        let mut out = vec![Fr::zero(); self.n() * (self.j as usize - 1)];
        ok(unsafe { h2v_extended_to_coeff(self.h, a.as_ptr() as *const u64, out.as_mut_ptr() as *mut u64) });
        out
    }
    pub fn divide_by_vanishing_poly(&self, a: &mut [Fr]) {
        assert_eq!(a.len(), self.extended_n());
        ok(unsafe { h2v_divide_by_vanishing_poly(self.h, a.as_mut_ptr() as *mut u64) })
    }
    /// `EvaluationDomain::rotate_omega(value, Rotation(rotation))`
    pub fn rotate_omega(&self, value: &Fr, rotation: i32) -> Fr {
        let mut out = Fr::zero();
        ok(unsafe { h2v_domain_rotate_omega(self.h, value as *const Fr as *const u64, rotation, &mut out as *mut Fr as *mut u64) });
        out
    }
    /// `EvaluationDomain::rotate_extended(&poly, Rotation(rotation))`
    pub fn rotate_extended(&self, poly: &[Fr], rotation: i32) -> Vec<Fr> {
        assert_eq!(poly.len(), self.extended_n());
        let mut out = vec![Fr::zero(); poly.len()];
        ok(unsafe { h2v_domain_rotate_extended(self.h, poly.as_ptr() as *const u64, rotation, out.as_mut_ptr() as *mut u64) });
        out
    }
    /// `EvaluationDomain::l_i_range(x, xn, lo..hi)`
    pub fn l_i_range(&self, x: &Fr, xn: &Fr, rotations: std::ops::Range<i32>) -> Vec<Fr> {
        let mut out = vec![Fr::zero(); rotations.len()];
        ok(unsafe { h2v_domain_l_i_range(self.h, x as *const Fr as *const u64, xn as *const Fr as *const u64, rotations.start, rotations.end,
                                         out.as_mut_ptr() as *mut u64) });
        out
    }
    fn fill(&self, basis: c_int, scalar: Option<&Fr>) -> Vec<Fr> {
        let mut out = vec![Fr::zero(); if basis == 2 { self.extended_n() } else { self.n() }];
        let p = scalar.map_or(std::ptr::null(), |s| s as *const Fr as *const u64);
        ok(unsafe { h2v_domain_fill(self.h, basis, p, out.as_mut_ptr() as *mut u64) });
        out
    }
    pub fn empty_coeff(&self) -> Vec<Fr> { self.fill(0, None) }
    pub fn empty_lagrange(&self) -> Vec<Fr> { self.fill(1, None) }
    pub fn empty_extended(&self) -> Vec<Fr> { self.fill(2, None) }
    pub fn constant_lagrange(&self, scalar: &Fr) -> Vec<Fr> { self.fill(1, Some(scalar)) }
    pub fn constant_extended(&self, scalar: &Fr) -> Vec<Fr> { self.fill(2, Some(scalar)) }
    /// `Evaluator::evaluate_h`, custom-gate loop for halo2-base's vertical gates, on device-resident extended columns
    /// (`d_q`, `d_a`: `n_gates` columns `stride` elements apart, from `h2v_domain_transform_dev(COEFF_TO_EXTENDED)`)
    pub fn quotient_gates(&self, d_h: *mut c_void, y: &Fr, n_gates: usize, d_q: *const c_void, d_a: *const c_void, stride: usize) {
        ok(unsafe { h2v_quotient_gates_dev(self.h, d_h, y as *const Fr as *const u64, n_gates, d_q, stride, d_a, stride) })
    }
    pub fn raw(&self) -> *mut H2vDomain { self.h }
}
impl Drop for DeviceDomain {
    fn drop(&mut self) { unsafe { h2v_domain_free(self.h) } }
}

/// A circuit recorded by a builder from `h2v_builder_new_recording`, replayed for batches of inputs on the device
/// (`witness_gen_only` for many inputs): `generate` gives each input's advice columns and instances, byte for byte what
/// the host builder and layouter give.  Inputs are the values the circuit passed to `assign_witnesses`, in order.
pub struct WitnessProgram { h: *mut H2vWitnessProgram, info: [u64; 8] }
unsafe impl Send for WitnessProgram {}
impl WitnessProgram {
    /// `recording` may be freed (`h2v_builder_free`) once this returns
    pub fn new(recording: *mut H2vBuilder, k: u32, minimum_rows: u32) -> Self {
        let mut h = std::ptr::null_mut();
        ok(unsafe { h2v_witness_program_new(recording, k, minimum_rows, &mut h) });
        let mut info = [0u64; 8];
        ok(unsafe { h2v_witness_program_info(h, info.as_mut_ptr()) });
        WitnessProgram { h, info }
    }
    pub fn n_inputs(&self) -> usize { self.info[0] as usize }
    /// inputs: one slice of n_inputs values per witness -> (advice columns, instances) per witness
    pub fn generate(&self, inputs: &[&[Fr]]) -> Vec<(Vec<Vec<Fr>>, Vec<Fr>)> {
        let (b, ni, na, nin, n) = (inputs.len(), self.n_inputs(), self.info[4] as usize, self.info[5] as usize, 1usize << self.info[6]);
        assert!(inputs.iter().all(|x| x.len() == ni));
        let flat: Vec<Fr> = inputs.iter().flat_map(|x| x.iter().copied()).collect();
        let mut adv = vec![Fr::zero(); b * na * n];
        let mut inst = vec![Fr::zero(); b * nin];
        ok(unsafe { h2v_witness_generate(self.h, b, ni, flat.as_ptr() as *const u64, adv.as_mut_ptr() as *mut u64, inst.as_mut_ptr() as *mut u64) });
        (0..b).map(|w| ((0..na).map(|c| adv[(w * na + c) * n..(w * na + c + 1) * n].to_vec()).collect(), inst[w * nin..(w + 1) * nin].to_vec()))
            .collect()
    }
}
impl Drop for WitnessProgram {
    fn drop(&mut self) { unsafe { h2v_witness_program_free(self.h) } }
}

/// A halo2 `ProvingKey` (fixed columns, permutation polynomials, constraint-system shape) resident on the device;
/// `create_proof` = halo2-axiom `plonk::create_proof::<KZGCommitmentScheme<Bn256>, ProverSHPLONK<_>, _, _, PoseidonTranscript<..>, _>`
/// for one circuit, as `gen_snark_shplonk` runs it (scaffold mod.rs:296).
pub struct DeviceProvingKey(*mut H2vPk);
unsafe impl Send for DeviceProvingKey {}
impl DeviceProvingKey {
    pub fn new(srs: &DeviceSrs, cs: &H2vCircuit, fixed: &[&[Fr]], sigma: &[&[Fr]], vk_transcript_repr: &Fr) -> Self {
        let n = 1usize << cs.k;
        assert!(fixed.len() == cs.n_fixed as usize && sigma.len() == cs.n_perm as usize);
        assert!(fixed.iter().chain(sigma.iter()).all(|c| c.len() == n));
        let f: Vec<*const u64> = fixed.iter().map(|c| c.as_ptr() as *const u64).collect();
        let s: Vec<*const u64> = sigma.iter().map(|c| c.as_ptr() as *const u64).collect();
        let mut h = std::ptr::null_mut();
        ok(unsafe { h2v_pk_load(srs.0, cs, f.as_ptr(), s.as_ptr(), vk_transcript_repr as *const Fr as *const u64, &mut h) });
        DeviceProvingKey(h)
    }
    /// advice: every advice column in Lagrange form (2^k values; the unusable rows are overwritten with blinding values);
    /// instances: the public inputs per instance column; returns the proof bytes (`transcript.finalize()`)
    pub fn create_proof(&self, n: usize, advice: &[&[Fr]], instances: &[&[Fr]], rng_seed: &[u8; 32]) -> Vec<u8> {
        assert!(advice.iter().all(|c| c.len() == n));
        let a: Vec<*const u64> = advice.iter().map(|c| c.as_ptr() as *const u64).collect();
        let i: Vec<*const u64> = instances.iter().map(|c| c.as_ptr() as *const u64).collect();
        let il: Vec<u32> = instances.iter().map(|c| c.len() as u32).collect();
        let mut out = vec![0u8; unsafe { h2v_proof_size(self.0) }];
        let mut len = 0usize;
        ok(unsafe { h2v_create_proof(self.0, a.as_ptr(), i.as_ptr(), il.as_ptr(), rng_seed.as_ptr(), out.as_mut_ptr(), out.len(), &mut len) });
        out.truncate(len);
        out
    }
    /// proof p = `create_proof(n, advice[p], instances[p], &rng_seeds[p])`, byte for byte; the proofs run in groups on the
    /// device, phase by phase (one vector-database query answered per proof)
    pub fn create_proofs(&self, n: usize, advice: &[&[&[Fr]]], instances: &[&[&[Fr]]], rng_seeds: &[[u8; 32]]) -> Vec<Vec<u8>> {
        let b = advice.len();
        assert!(instances.len() == b && rng_seeds.len() == b);
        assert!(advice.iter().all(|a| a.iter().all(|c| c.len() == n)));
        let a: Vec<Vec<*const u64>> = advice.iter().map(|a| a.iter().map(|c| c.as_ptr() as *const u64).collect()).collect();
        let i: Vec<Vec<*const u64>> = instances.iter().map(|a| a.iter().map(|c| c.as_ptr() as *const u64).collect()).collect();
        let il: Vec<Vec<u32>> = instances.iter().map(|a| a.iter().map(|c| c.len() as u32).collect()).collect();
        let ap: Vec<*const *const u64> = a.iter().map(|v| v.as_ptr()).collect();
        let ip: Vec<*const *const u64> = i.iter().map(|v| v.as_ptr()).collect();
        let lp: Vec<*const u32> = il.iter().map(|v| v.as_ptr()).collect();
        let seeds: Vec<u8> = rng_seeds.iter().flatten().copied().collect();
        let size = unsafe { h2v_proof_size(self.0) };
        let mut out = vec![0u8; b * size];
        if b > 0 {
            ok(unsafe { h2v_create_proofs(self.0, b, ap.as_ptr(), ip.as_ptr(), lp.as_ptr(), seeds.as_ptr(), out.as_mut_ptr(), size) });
        }
        out.chunks(size.max(1)).take(b).map(|c| c.to_vec()).collect()
    }
    /// result w = `mock_prover(cs, fixed, sigma, advice[w], instances[w], max_failures)` with this key's circuit and
    /// columns; one device call for the batch, the key-only work done once per key
    pub fn mock_prover(&self, n: usize, advice: &[&[&[Fr]]], instances: &[&[&[Fr]]], max_failures: usize) -> Vec<(Vec<H2vMockFailure>, u64)> {
        let b = advice.len();
        assert!(instances.len() == b);
        assert!(advice.iter().all(|a| a.iter().all(|c| c.len() == n)));
        let a: Vec<Vec<*const u64>> = advice.iter().map(|a| a.iter().map(|c| c.as_ptr() as *const u64).collect()).collect();
        let i: Vec<Vec<*const u64>> = instances.iter().map(|a| a.iter().map(|c| c.as_ptr() as *const u64).collect()).collect();
        let il: Vec<Vec<u32>> = instances.iter().map(|a| a.iter().map(|c| c.len() as u32).collect()).collect();
        let ap: Vec<*const *const u64> = a.iter().map(|v| v.as_ptr()).collect();
        let ip: Vec<*const *const u64> = i.iter().map(|v| v.as_ptr()).collect();
        let lp: Vec<*const u32> = il.iter().map(|v| v.as_ptr()).collect();
        let mut out = vec![H2vMockFailure::default(); b * max_failures];
        let mut totals = vec![0u64; b];
        if b > 0 {
            ok(unsafe { h2v_pk_mock_prover(self.0, b, ap.as_ptr(), ip.as_ptr(), lp.as_ptr(), out.as_mut_ptr(), max_failures, totals.as_mut_ptr()) });
        }
        (0..b).map(|w| (out[w * max_failures..w * max_failures + (totals[w] as usize).min(max_failures)].to_vec(), totals[w])).collect()
    }
    /// `create_proofs` on the columns `program.generate(inputs)` gives, generated in this key's workspace on the device
    /// without crossing to the host -> (proof, instances) per input
    pub fn create_proofs_from_inputs(&self, program: &WitnessProgram, inputs: &[&[Fr]], rng_seeds: &[[u8; 32]]) -> Vec<(Vec<u8>, Vec<Fr>)> {
        let (b, ni, nin) = (inputs.len(), program.n_inputs(), program.info[5] as usize);
        assert!(rng_seeds.len() == b && inputs.iter().all(|x| x.len() == ni));
        let flat: Vec<Fr> = inputs.iter().flat_map(|x| x.iter().copied()).collect();
        let seeds: Vec<u8> = rng_seeds.iter().flatten().copied().collect();
        let size = unsafe { h2v_proof_size(self.0) };
        let mut out = vec![0u8; b * size];
        let mut inst = vec![Fr::zero(); b * nin];
        if b > 0 {
            ok(unsafe { h2v_create_proofs_from_inputs(self.0, program.h, b, ni, flat.as_ptr() as *const u64, seeds.as_ptr(), out.as_mut_ptr(), size,
                                                      inst.as_mut_ptr() as *mut u64) });
        }
        (0..b).map(|p| (out[p * size..(p + 1) * size].to_vec(), inst[p * nin..(p + 1) * nin].to_vec())).collect()
    }
    /// `mock_prover` on the same generated columns, one device call for the batch
    pub fn mock_prover_from_inputs(&self, program: &WitnessProgram, inputs: &[&[Fr]], max_failures: usize) -> Vec<(Vec<H2vMockFailure>, u64)> {
        let (b, ni) = (inputs.len(), program.n_inputs());
        assert!(inputs.iter().all(|x| x.len() == ni));
        let flat: Vec<Fr> = inputs.iter().flat_map(|x| x.iter().copied()).collect();
        let mut out = vec![H2vMockFailure::default(); b * max_failures];
        let mut totals = vec![0u64; b];
        if b > 0 {
            ok(unsafe { h2v_pk_mock_prover_from_inputs(self.0, program.h, b, ni, flat.as_ptr() as *const u64, out.as_mut_ptr(), max_failures,
                                                       totals.as_mut_ptr()) });
        }
        (0..b).map(|w| (out[w * max_failures..w * max_failures + (totals[w] as usize).min(max_failures)].to_vec(), totals[w])).collect()
    }
}
impl Drop for DeviceProvingKey {
    fn drop(&mut self) { unsafe { h2v_pk_free(self.0) } }
}
