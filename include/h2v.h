/*
 * h2v.h -- C ABI of libh2v.so: the B200 (sm_100a) backend for the KZG-commit and
 * EvaluationDomain hot path underneath erhant/halo2-vectordb's keygen / prove flow.
 *
 * The reference has no FFI seam on this path: its scaffold (/root/reference/src/scaffold/mod.rs:273
 * create_pk, :296 gen_snark_shplonk) calls in-process Rust generics of the un-vendored halo2-axiom
 * crate (Cargo.toml:19-28).  Each entry point below names the upstream function a patched
 * halo2-axiom would forward to it (SURVEY.md 8(a)/(b)); INTEGRATION.md shows the Rust binding.
 *
 * Conventions (identical to halo2curves bn256, so Rust slices cross the boundary by pointer):
 *   Fr / Fq element   4 x uint64_t little-endian limbs, MONTGOMERY form (R = 2^256)      32 B
 *   G1Affine          {x, y} Fq                       identity = (0, 0)                  64 B
 *   G1 (Jacobian)     {x, y, z} Fq                    identity z = 0                     96 B
 * All pointers are HOST pointers unless the parameter name starts with `d_`.
 * Return value: 0 on success, a negative H2V_E* code otherwise; h2v_last_error() (thread-local)
 * describes the failure.  There is NO CPU fallback: without a usable CUDA device every compute
 * entry point fails with H2V_ECUDA.  Entry points are thread-safe; calls on one handle serialise.
 * One process drives one or several GPUs (h2v_init): polynomial columns are partitioned across the devices, each
 * of which holds an SRS replica (SURVEY.md 8(e)); no collective is needed.  One process per GPU works as well.
 */
#ifndef H2V_H
#define H2V_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define H2V_OK 0
#define H2V_EINVAL (-1)   /* bad argument (the reference would panic on the same input: assert_eq!(len, 1 << log_n) etc.) */
#define H2V_ECUDA (-2)    /* CUDA runtime error or no device */
#define H2V_ENOMEM (-3)

#define H2V_BASIS_MONOMIAL 0 /* ParamsKZG::g          -> commit          */
#define H2V_BASIS_LAGRANGE 1 /* ParamsKZG::g_lagrange -> commit_lagrange */

typedef struct h2v_srs *h2v_srs_t;       /* device-resident ParamsKZG bases (+ window tables) */
typedef struct h2v_domain *h2v_domain_t; /* EvaluationDomain: constants + device twiddles      */

/* ---- runtime ------------------------------------------------------------------------------ */
/* The CUDA devices this process drives, in order (SURVEY.md 8(b)); devices[0] is the primary device.  Every handle
 * created afterwards holds one replica per listed device (the SRS window tables are built on the primary device and
 * copied device to device once); `_dev` entry points run on the device that owns their buffers; the host-facing batch
 * entry points (h2v_commit_batch, h2v_domain_transform_batch) send column j to device j mod n_dev -- each device pulls
 * its columns over its own PCIe link, no collective -- and return results in column order; everything else runs on the
 * primary device.  Call once, before creating handles; NULL / 0 selects device 0 (the default without a call).
 * Mirrors nothing upstream: the reference is CPU-only and single-process (scaffold mod.rs:251-323). */
int h2v_init(const int *devices, int n_dev);
/* the device list in use; returns its length */
int h2v_device_list(int *out, int cap);
int h2v_device_count(void);
const char *h2v_last_error(void);
const char *h2v_version(void);

/* Device buffers for the `_dev` entry points (columns that stay in HBM between commit / transform / evaluation
 * steps of one prover phase); plain synchronous copies. */
int h2v_dev_alloc(size_t bytes, void **d_out);                       /* on the primary device */
int h2v_dev_alloc_on(int device, size_t bytes, void **d_out);        /* on one of the h2v_init devices */
int h2v_dev_free(void *d_ptr);
int h2v_dev_upload(void *d_dst, const void *src, size_t bytes);
int h2v_dev_download(void *dst, const void *d_src, size_t bytes);
/* Page-lock a caller-owned buffer (a Rust Vec<Fr>, a numpy array) so that the library's asynchronous,
 * double-buffered H2D / D2H copies really overlap with the kernels; pageable memory works too, only slower. */
int h2v_host_register(void *ptr, size_t bytes);
int h2v_host_unregister(void *ptr);

/* ---- KZG commit path ---------------------------------------------------------------------- */
/* halo2-axiom poly/kzg/commitment.rs ParamsKZG {k, n, g, g_lagrange}: upload both bases
 * (n = 2^k G1Affine each) and build the per-window tables 2^(jc) * B_i once.
 * `g` or `g_lagrange` may be NULL if that basis is never used.  (scaffold: gen_srs, mod.rs:260) */
int h2v_srs_load(uint32_t k, const uint64_t *g, const uint64_t *g_lagrange, h2v_srs_t *out);
/* ParamsKZG::setup(k, rng) with the secret supplied by the caller (upstream draws s = Fr::random(rng); gen_srs
 * seeds ChaCha20 with zeros -- "unsafe" by design): g[i] = s^i G and g_lagrange[i] = L_i(s) G, each 2^k affine
 * points (either output may be NULL).  One-time work; g2 / s_g2 are verifier-side and not produced. */
int h2v_srs_setup(uint32_t k, const uint64_t s_mont[4], uint64_t *g_out, uint64_t *g_lagrange_out);
/* halo2-base gen_srs(k)'s setup branch (scaffold mod.rs:260): ParamsKZG::setup(k, ChaCha20Rng::from_seed(seed)) -- the
 * secret is the generator's first Fr::random draw (seed = 32 zero bytes upstream: "unsafe" by design).  Outputs (each may
 * be NULL): g, g_lagrange (2^k affine points, computed on the device), g2 = the G2 generator and s_g2 = s * g2 (G2Affine:
 * x.c0, x.c1, y.c0, y.c1 Montgomery Fq, 128 bytes; host-side). */
int h2v_srs_gen(uint32_t k, const uint8_t seed[32], uint64_t *g_out, uint64_t *g_lagrange_out, uint64_t g2_out[16], uint64_t s_g2_out[16]);
int h2v_g2_mul_generator(const uint64_t s_mont[4], uint64_t out[16]);
/* ParamsKZG::write / read, SerdeFormat::RawBytes (params/kzg_bn254_{k}.srs): k as u32 LE, g, g_lagrange, g2, s_g2 as raw
 * Montgomery limbs.  read: *k_out always receives the file's k; buffers must hold cap_points >= 2^k points each. */
int h2v_srs_write_file(const char *path, uint32_t k, const uint64_t *g, const uint64_t *g_lagrange, const uint64_t g2[16],
                       const uint64_t s_g2[16]);
int h2v_srs_read_file(const char *path, uint32_t *k_out, uint64_t *g, uint64_t *g_lagrange, size_t cap_points, uint64_t g2[16],
                      uint64_t s_g2[16]);
void h2v_srs_free(h2v_srs_t srs);
/* window size c and number of windows W = ceil(255 / c) of the table the handle's last commit used (diagnostics) */
int h2v_srs_info(h2v_srs_t srs, uint32_t *window_bits, uint32_t *windows);
/* ParamsKZG::commit(poly, _blind) / commit_lagrange(poly, _blind) = best_multiexp(poly, bases[..len]);
 * the Blind argument is ignored by KZG upstream, so it is not part of the ABI.  len <= 2^k.
 * Output: the unique affine representative (G1::to_affine()). */
int h2v_commit(h2v_srs_t srs, int basis, const uint64_t *poly, size_t len, uint64_t out_affine[8]);
/* The same for `n_polys` columns in one call (create_proof commits every advice / lookup /
 * permutation column against the same bases; this is the preferred entry point). polys[i] -> len Fr. */
int h2v_commit_batch(h2v_srs_t srs, int basis, const uint64_t *const *polys, size_t n_polys, size_t len,
                     uint64_t *out_affine /* n_polys x 8 */);
/* Device-resident variant: d_polys = n_polys columns of `len` Fr, `col_stride` elements apart;
 * d_out_affine = n_polys x 64 B on the device.  Asynchronous work is complete on return. */
int h2v_commit_batch_dev(h2v_srs_t srs, int basis, const void *d_polys, size_t col_stride, size_t n_polys, size_t len,
                         void *d_out_affine);
/* The advice phase of create_proof in one call: host columns that are committed AND left resident.  Column j is uploaded,
 * its rows [row0, row0 + n_rows) are overwritten with tails[j * n_rows ...] (the blinding rows; n_rows may be 0), it is
 * committed, and it is stored at d_dst + j * dst_stride (Fr elements; a buffer on one of the h2v_init devices).  With
 * several devices the columns are cut into contiguous blocks: every device uploads its block over its own PCIe link,
 * commits it against its SRS replica and forwards it to d_dst over NVLink.  out_affine: n_polys host G1Affine. */
int h2v_commit_batch_resident(h2v_srs_t srs, int basis, const uint64_t *const *polys, size_t n_polys, size_t len, const uint64_t *tails,
                              size_t row0, size_t n_rows, void *d_dst, size_t dst_stride, uint64_t *out_affine);
/* halo2-axiom arithmetic.rs best_multiexp(coeffs, bases) -> C::Curve, exact shape: arbitrary bases,
 * no handle, Jacobian result (any representative; compare after to_affine). */
int h2v_best_multiexp(const uint64_t *coeffs, const uint64_t *bases, size_t n, uint64_t out_jacobian[12]);
/* sum of n affine points, affine result: the fold of the per-thread partial sums at the end of best_multiexp
 * (arithmetic.rs: `results.iter().fold(C::Curve::identity(), |a, b| a + b)`), used here to combine the per-GPU
 * partial sums of ONE multiexp whose index range was split across GPUs (SURVEY.md 8(e), config 5). */
int h2v_g1_sum(const uint64_t *affine_pts, size_t n, uint64_t out_affine[8]);

/* ---- EvaluationDomain --------------------------------------------------------------------- */
/* arithmetic.rs best_fft(a, omega, log_n): in place, natural order in and out. */
int h2v_best_fft(uint64_t *a, const uint64_t omega[4], uint32_t log_n);
/* poly/domain.rs EvaluationDomain::new(j, k) */
int h2v_domain_new(uint32_t j, uint32_t k, h2v_domain_t *out);
void h2v_domain_free(h2v_domain_t dom);
uint32_t h2v_domain_k(h2v_domain_t dom);
uint32_t h2v_domain_extended_k(h2v_domain_t dom);
/* scalar getters: 0 omega, 1 omega_inv, 2 extended_omega, 3 extended_omega_inv, 4 g_coset, 5 g_coset_inv,
 * 6 ifft_divisor, 7 extended_ifft_divisor, 8+i t_evaluations[i] */
int h2v_domain_constant(h2v_domain_t dom, int which, uint64_t out[4]);
/* EvaluationDomain::rotate_omega(value, Rotation(rotation)) = value * omega^rotation (host-side scalar helper) */
int h2v_domain_rotate_omega(h2v_domain_t dom, const uint64_t value[4], int32_t rotation, uint64_t out[4]);
/* EvaluationDomain::rotate_extended(poly, Rotation(rotation)): out[i] = in[(i + rotation * 2^(extended_k - k)) mod 2^extended_k];
 * host columns of 2^extended_k Fr, in != out */
int h2v_domain_rotate_extended(h2v_domain_t dom, const uint64_t *in, int32_t rotation, uint64_t *out);
/* EvaluationDomain::l_i_range(x, xn, rot_lo..rot_hi): out[t] = l_{rot_lo + t}(x), the Lagrange basis polynomials of the
 * 2^k domain at x (xn = x^n supplied by the caller, as upstream's verifier does) */
int h2v_domain_l_i_range(h2v_domain_t dom, const uint64_t x[4], const uint64_t xn[4], int32_t rot_lo, int32_t rot_hi, uint64_t *out);
/* EvaluationDomain::{empty_coeff, empty_lagrange, empty_extended, constant_lagrange, constant_extended}: fill a host column
 * of the basis' length with `scalar` (NULL = zero); basis 0 coeff, 1 lagrange (2^k each), 2 extended (2^extended_k) */
int h2v_domain_fill(h2v_domain_t dom, int basis, const uint64_t scalar[4], uint64_t *out);
/* EvaluationDomain::lagrange_to_coeff / coeff_to_lagrange (private fft/ifft on the 2^k domain); in place */
int h2v_lagrange_to_coeff(h2v_domain_t dom, uint64_t *a);
int h2v_coeff_to_lagrange(h2v_domain_t dom, uint64_t *a);
/* EvaluationDomain::coeff_to_extended: in 2^k, out 2^extended_k */
int h2v_coeff_to_extended(h2v_domain_t dom, const uint64_t *in, uint64_t *out);
/* EvaluationDomain::extended_to_coeff: in 2^extended_k, out 2^k * (j-1) */
int h2v_extended_to_coeff(h2v_domain_t dom, const uint64_t *in, uint64_t *out);
/* EvaluationDomain::divide_by_vanishing_poly: in place on 2^extended_k */
int h2v_divide_by_vanishing_poly(h2v_domain_t dom, uint64_t *a);
/* batched over independent columns (host pointers, one per column) */
#define H2V_OP_LAGRANGE_TO_COEFF 0
#define H2V_OP_COEFF_TO_LAGRANGE 1
#define H2V_OP_COEFF_TO_EXTENDED 2
#define H2V_OP_EXTENDED_TO_COEFF 3
#define H2V_OP_DIVIDE_BY_VANISHING 4 /* fused: divide_by_vanishing_poly then extended_to_coeff */
int h2v_domain_transform_batch(h2v_domain_t dom, int op, const uint64_t *const *in, uint64_t *const *out, size_t n_cols);
/* device-resident: columns `in_stride` / `out_stride` elements apart; d_in != d_out */
int h2v_domain_transform_dev(h2v_domain_t dom, int op, const void *d_in, size_t in_stride, void *d_out, size_t out_stride,
                             size_t n_cols);

/* ---- polynomial primitives around the commits ("next": SURVEY.md 8(f) row 2) ------------------ */
/* arithmetic.rs eval_polynomial(poly, point) for every (poly, point) pair: out[p * n_points + t] */
int h2v_eval_polynomial_batch(const uint64_t *const *polys, size_t n_polys, size_t len, const uint64_t *points, size_t n_points,
                              uint64_t *out);
int h2v_eval_polynomial_dev(const void *d_polys, size_t stride, size_t n_polys, size_t len, const void *d_points, size_t n_points,
                            void *d_out);
/* ff BatchInvert::batch_invert: every non-zero element replaced by its inverse, zeros untouched; in place */
int h2v_batch_invert(uint64_t *a, size_t n);
/* running product of the permutation / lookup arguments: out[0] = 1, out[i+1] = out[i] * num[i] / den[i] (den != 0) */
int h2v_grand_product(const uint64_t *num, const uint64_t *den, size_t n, uint64_t *out);
/* the same for n_cols device-resident columns, contiguous (n elements apart): one batch inversion for all of them */
int h2v_grand_product_dev(const void *d_num, const void *d_den, size_t n, size_t n_cols, void *d_out);
/* arithmetic.rs kate_division(a, b): quotient of a(X) (n coefficients) by (X - b), n - 1 coefficients */
int h2v_kate_division(const uint64_t *a, size_t n, const uint64_t b[4], uint64_t *out);
int h2v_kate_division_dev(const void *d_a, size_t n, const uint64_t b[4], void *d_out /* n - 1, no overlap with d_a */);

/* halo2-axiom plonk/lookup/prover.rs permute_expression_pair [UPSTREAM] (create_proof step 5): from the first
 * `usable_rows` values of the compressed input and table expressions, permuted_input = the input sorted ascending
 * (canonical integers) and permuted_table = the table rearranged so that permuted_table[i] == permuted_input[i] on every
 * row where permuted_input changes, the leftover table values filling the repeated rows (ascending values onto the
 * repeated rows taken from the last one backwards, as upstream's `pop()` does).  H2V_EINVAL when an input value is
 * not in the table (upstream: Error::ConstraintSystemFailure).  The caller appends the blinding rows. */
int h2v_permute_expression_pair(const uint64_t *input, const uint64_t *table, size_t usable_rows, uint64_t *permuted_input,
                                uint64_t *permuted_table);
int h2v_permute_expression_pair_dev(const void *d_input, const void *d_table, size_t usable_rows, void *d_permuted_input,
                                    void *d_permuted_table);
/* every lookup argument of one proof phase in one set of launches: d_inputs[l] / d_tables[l] are device columns (a table
 * shared by several lookups is sorted once), the permuted columns land at d_permuted_inputs + l * input_stride and
 * d_permuted_tables + l * table_stride (strides in elements) */
int h2v_permute_expression_pair_batch_dev(const void *const *d_inputs, const void *const *d_tables, size_t n_lookups, size_t usable_rows,
                                          void *d_permuted_inputs, size_t input_stride, void *d_permuted_tables, size_t table_stride);

/* ---- quotient evaluation on the extended coset ("next": SURVEY.md 8(f) row 1) ------------------------------
 * The per-row loops of halo2-axiom plonk/evaluation.rs Evaluator::evaluate_h [UPSTREAM; reached from
 * src/scaffold/mod.rs:296] for the constraint system halo2-base builds.  Every polynomial is a device-resident
 * column of 2^extended_k Fr values (h2v_dev_alloc; produced by h2v_domain_transform_dev COEFF_TO_EXTENDED), so the
 * 4n-sized columns never cross PCIe; `d_h` is the running value, updated in place as  h <- h * y + term  for each
 * term in upstream's order (custom gates, then permutation, then each lookup).  Start from a zeroed column and
 * finish with h2v_domain_transform_dev(H2V_OP_DIVIDE_BY_VANISHING).  Rotation r reads row i + r * 2^(extended_k-k). */
/* custom gates: halo2-base's vertical gate on advice column j,  q_j * (a_j + a_j(wX) * a_j(w^2 X) - a_j(w^3 X)) */
int h2v_quotient_gates_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], size_t n_gates, const void *d_q, size_t q_stride,
                           const void *d_a, size_t a_stride);
/* the same with the selector / advice columns given as device-resident tables of n_gates column pointers (the prover's
 * columns live in different allocations: fixed columns in the proving key, advice columns in the proof workspace) */
int h2v_quotient_gates_ptrs_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], size_t n_gates, const void *const *d_q_ptrs,
                                const void *const *d_a_ptrs);
/* permutation argument: `n_cols` permuted columns (advice / fixed / instance values, in permutation-column order) with
 * their sigma polynomials, ceil(n_cols / chunk_len) grand products z (chunk_len = cs.degree() - 2), l_0, l_last and
 * l_active_row; X = g_coset * extended_omega^i and Fr::DELTA come from the domain. */
int h2v_quotient_permutation_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                 size_t n_cols, size_t chunk_len, const void *d_cols, size_t cols_stride, const void *d_sigma,
                                 size_t sigma_stride, const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last,
                                 const void *d_l_active, uint32_t blinding_factors);
int h2v_quotient_permutation_ptrs_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                      size_t n_cols, size_t chunk_len, const void *const *d_col_ptrs, const void *const *d_sigma_ptrs,
                                      const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last, const void *d_l_active,
                                      uint32_t blinding_factors);
/* the same argument folded in slices, for proofs whose extended columns do not all fit in HBM at once (k = 20): this call
 * folds the terms that precede the per-set products when `with_head` is set (they read every z), then the products of the
 * sets [set_begin, set_end); the two pointer tables hold only the columns of those sets (entry 0 = column
 * set_begin * chunk_len).  Calls with with_head = 1 on the first slice and consecutive set ranges give exactly the
 * result of one h2v_quotient_permutation_ptrs_dev call. */
int h2v_quotient_permutation_range_ptrs_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                            size_t n_cols, size_t chunk_len, size_t set_begin, size_t set_end, int with_head,
                                            const void *const *d_col_ptrs, const void *const *d_sigma_ptrs, const void *d_z, size_t z_stride,
                                            const void *d_l0, const void *d_l_last, const void *d_l_active, uint32_t blinding_factors);
/* one lookup argument: compressed input / table expressions (theta-folded by the caller; for halo2-base's range
 * lookup they are the lookup advice column and the fixed table column), permuted A' / S', grand product z */
int h2v_quotient_lookup_dev(h2v_domain_t dom, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                            const void *d_input, const void *d_table, const void *d_perm_input, const void *d_perm_table,
                            const void *d_z, const void *d_l0, const void *d_l_last, const void *d_l_active);

/* ---- create_proof ("next": SURVEY.md 8(f) rows 2-3) ---------------------------------------------------------
 * One Halo2-KZG (SHPLONK) proof of one circuit, restating halo2-axiom plonk/prover.rs create_proof [UPSTREAM] as reached
 * from /root/reference/src/scaffold/mod.rs:296 (gen_snark_shplonk) with the transcript of mod.rs:309-310.  The constraint
 * system must have the shape halo2-base builds (one vertical gate per basic-gate advice column, single-expression range
 * lookups, a permutation over any columns); witness generation and keygen stay with the caller (the Rust side), which
 * hands over what halo2's ProvingKey holds. */
typedef struct {
    uint32_t k;                 /* 2^k rows */
    uint32_t degree;            /* cs.degree(): EvaluationDomain::new(degree, k); permutation chunk = degree - 2 */
    uint32_t blinding_factors;  /* cs.blinding_factors(): the last blinding_factors + 1 rows of every column are unusable */
    uint32_t n_advice, n_fixed, n_instance;
    uint32_t n_gates;           /* gate j: fixed[gate_selector[j]] * (a + a(wX) a(w^2 X) - a(w^3 X)), a = advice[gate_advice[j]] */
    const uint32_t *gate_advice, *gate_selector;
    uint32_t n_lookups;         /* lookup l: advice[lookup_input[l]] must lie in fixed[lookup_table[l]] */
    const uint32_t *lookup_input, *lookup_table;
    uint32_t n_perm;            /* cs.permutation.columns in order: kind 0 advice, 1 fixed, 2 instance */
    const uint8_t *perm_kind;
    const uint32_t *perm_index;
    uint32_t n_advice_queries;  /* cs.advice_queries in order: (column, rotation) */
    const uint32_t *advice_query_col;
    const int32_t *advice_query_rot;
    uint32_t n_fixed_queries;   /* cs.fixed_queries in order */
    const uint32_t *fixed_query_col;
    const int32_t *fixed_query_rot;
} h2v_circuit_t;
typedef struct h2v_pk *h2v_pk_t; /* ProvingKey: fixed / sigma polynomials in Lagrange, coefficient and extended form, resident */
/* fixed: pk.fixed_values (n_fixed Lagrange columns of 2^k); sigma: pk.permutation.permutations (n_perm Lagrange columns);
 * vk_transcript_repr: vk.transcript_repr (upstream hashes the pinned verifying key's Debug text; the caller supplies it).
 * The srs handle must outlive the pk and hold both bases. */
int h2v_pk_load(h2v_srs_t srs, const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma,
                const uint64_t vk_transcript_repr[4], h2v_pk_t *out);
void h2v_pk_free(h2v_pk_t pk);
/* advice: n_advice Lagrange columns of 2^k (the unusable rows are overwritten with blinding values); instances[c]: the
 * instance_len[c] public inputs of instance column c; rng_seed: ChaCha20Rng::from_seed.  Writes the proof (the transcript's
 * byte stream, exactly h2v_proof_size(pk) bytes) to proof_out. */
int h2v_create_proof(h2v_pk_t pk, const uint64_t *const *advice, const uint64_t *const *instances, const uint32_t *instance_len,
                     const uint8_t rng_seed[32], uint8_t *proof_out, size_t proof_cap, size_t *proof_len);
/* n_proofs proofs on one key: proof p = h2v_create_proof(pk, advice[p], instances[p], instance_len[p], rng_seeds + 32 p),
 * written to proofs_out + p * proof_stride (proof_stride >= h2v_proof_size(pk)).  Byte for byte the proofs of n_proofs
 * h2v_create_proof calls; the proofs run in groups, phase by phase, so that each launch, commit and synchronisation is
 * paid once per group.  Group size: H2V_PROOF_GROUP if set, else as many proofs as fit in the device memory the key
 * leaves (8 GB kept free); a group that runs out of memory is halved; streamed keys prove one at a time.  Every proof's
 * inputs are checked before any device work; an error text names the proof it concerns ("create_proofs: proof 2: ...")
 * and the key stays usable.  n_proofs = 0 does nothing.  Calls on one key serialise. */
int h2v_create_proofs(h2v_pk_t pk, size_t n_proofs, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
                      const uint32_t *const *instance_len, const uint8_t *rng_seeds, uint8_t *proofs_out, size_t proof_stride);
size_t h2v_proof_size(h2v_pk_t pk);
/* wall-clock milliseconds per phase of the last h2v_create_proof / h2v_create_proofs call on this key, summed over the
 * call's groups: 0 upload + advice commitments, 1 lookup permutations, 2 grand products, 3 random polynomial +
 * transforms, 4 evaluate_h + quotient commitments, 5 evaluations, 6 multi-open argument; out[7]: the number of groups
 * the call ran in */
int h2v_pk_last_phase_ms(h2v_pk_t pk, double out[8]);

/* ---- mock prover: check a laid-out circuit's constraints -------------------------------------------------------
 * halo2 `MockProver::run(k, circuit, instances).assert_satisfied()` (the reference's `mock` command, scaffold mod.rs:263)
 * for the constraint-system shape above, on the primary device.  The inputs are those of h2v_pk_load + h2v_create_proof:
 * Lagrange columns of 2^k in Montgomery form; no SRS and no key.  Values are compared as field elements (limbs that are
 * not reduced compare equal to their reduced form).
 *   gates        gate j, every row with fixed[gate_selector[j]][row] != 0: GATE_UNUSABLE if row + 3 >= usable rows
 *                (2^k - blinding_factors - 1), else GATE if a + a(w) a(w^2) - a(w^3) != 0.  column = j, other_column = the
 *                gate's advice column, other_row = row.
 *   lookups      lookup l, every usable row: advice[lookup_input[l]][row] must occur among the usable rows of
 *                fixed[lookup_table[l]]; else LOOKUP with column = l, other_column = the input column, other_row = row.
 *   permutation  permutation column c, every row: sigma[c][row] must be delta^c2 * w^r2 with c2 < n_perm, else
 *                SIGMA_NOT_DELTA_OMEGA (other_column = other_row = 0xFFFFFFFF) and the cell's other checks are skipped;
 *                SIGMA_NOT_PERMUTATION when a cell earlier in (column, row) order has the same image; when the image is
 *                another cell, COPY_UNUSABLE if either row is unusable and COPY if the two cell values differ.  Instance
 *                column c holds instances[c] in its first instance_len[c] rows and zeros below.  column / row = (c, row),
 *                other_column / other_row = (c2, r2).
 * failures_out receives the first min(cap, total) failures in this order: gates, lookups, permutation; then by gate,
 * lookup or permutation column; then by row; within one cell SIGMA_NOT_DELTA_OMEGA, SIGMA_NOT_PERMUTATION,
 * COPY_UNUSABLE, COPY.  *n_failures = the exact total.  The same inputs always give the same output.
 * Every argument is checked before any device work (H2V_EINVAL: NULL pointers, the column indices of cs as h2v_pk_load
 * checks them, instance_len[c] > 2^k, more than 65535 gates / lookups / permutation columns, more than 2^32 flags).
 * Device memory: the columns (32 bytes per cell of every advice, fixed, sigma and instance column), 8 bytes per
 * permutation cell, one bit per gate row, lookup row and 8 per permutation cell, the table of the 2^k values w^r (40 bytes
 * per row) and the sorted lookup tables (32 bytes per row and distinct table): about 31 GB for the SIFT-shaped k = 20
 * circuit (28.3 GB of columns, 290 permutation columns). */
typedef struct {
    uint32_t kind, column, row, other_column, other_row;
} h2v_mock_failure_t;
enum {
    H2V_MOCK_GATE = 1, H2V_MOCK_GATE_UNUSABLE, H2V_MOCK_LOOKUP, H2V_MOCK_SIGMA_NOT_DELTA_OMEGA, H2V_MOCK_SIGMA_NOT_PERMUTATION,
    H2V_MOCK_COPY_UNUSABLE, H2V_MOCK_COPY
};
int h2v_mock_prover(const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma, const uint64_t *const *advice,
                    const uint64_t *const *instances, const uint32_t *instance_len, h2v_mock_failure_t *failures_out, size_t cap,
                    uint64_t *n_failures);
/* The mock prover on a loaded key, for n_witnesses witnesses in one call: with cs, fixed and sigma what h2v_pk_load
 * received, failures_out + w * cap receives what h2v_mock_prover(cs, fixed, sigma, advice[w], instances[w],
 * instance_len[w], ., cap, .) writes, and n_failures[w] that call's exact total (same order, same fields, same cap).
 * Only the witnesses are uploaded, into the key's proof workspace.  What depends on the key alone (each sigma cell
 * decoded into its image, the permutation's key-only failures, the sorted lookup tables: about 4.5 bytes per permutation
 * cell and 32 bytes per row and distinct table) is built by the first call and kept with the key until h2v_pk_free.
 * The witnesses run in groups, as h2v_create_proofs runs proofs (H2V_PROOF_GROUP if set, else as many as fit with 8 GB
 * kept free; a group that runs out of memory is halved).  Every argument is checked before any device work, as
 * h2v_mock_prover checks it; an error text names the witness it concerns ("pk_mock_prover: witness 2: ...") and the key
 * stays usable.  The call writes none of the key's columns: proofs made after it are unchanged.  n_witnesses = 0 does
 * nothing.  Calls on one key serialise with its proofs. */
int h2v_pk_mock_prover(h2v_pk_t pk, size_t n_witnesses, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
                       const uint32_t *const *instance_len, h2v_mock_failure_t *failures_out, size_t cap, uint64_t *n_failures);
/* wall-clock milliseconds of the calling thread's last h2v_mock_prover or h2v_pk_mock_prover call: out[0] the upload of
 * the columns (h2v_pk_mock_prover: the witnesses' columns), out[1] the checks (building the key tables -- for
 * h2v_pk_mock_prover on the key's first call only --, every kernel, the compaction and the download of the failures) */
int h2v_mock_last_ms(double out[2]);

/* ---- circuit builder ("next": SURVEY.md 8(f) row 4; host-side, no device needed) -----------------------------------
 * The step before the hot path: the reference's chips produce the execution trace whose columns create_proof commits.
 * One builder = halo2-base's GateThreadBuilder with the single Context the scaffold uses (`builder.main(0)`,
 * /root/reference/src/scaffold/mod.rs:61) plus FixedPointChip<Fr, PRECISION_BITS>::default(lookup_bits)
 * (/root/reference/src/gadget/fixed_point.rs:100), DistanceChip::default and VectorDBChip::default over it.
 * Cells are named by their offset in the trace (AssignedValue); values cross the ABI in Montgomery form.
 * Upstream panics (asserts, division by zero, index out of range) return H2V_EINVAL with the panic text. */
typedef struct h2v_builder *h2v_builder_t;
typedef struct h2v_layout *h2v_layout_t;
enum {
    /* FixedPointInstructions (fixed_point.rs:217-467), two cells in -> one cell out */
    H2V_FP_QADD = 1, H2V_FP_QSUB, H2V_FP_QMUL, H2V_FP_QDIV, H2V_FP_QMOD, H2V_FP_QPOW, H2V_FP_QMAX, H2V_FP_QMIN, H2V_FP_BIT_XOR,
    H2V_FP_COND_NEG, /* (a, is_neg) */
    /* one cell in -> one cell out */
    H2V_FP_NEG = 20, H2V_FP_QABS, H2V_FP_IS_NEG, H2V_FP_SIGN, H2V_FP_CLIP, H2V_FP_QEXP2, H2V_FP_QLOG2, H2V_FP_QEXP, H2V_FP_QLOG,
    H2V_FP_QSQRT, H2V_FP_QSIN, H2V_FP_QCOS, H2V_FP_QTAN, H2V_FP_QSINH, H2V_FP_QCOSH, H2V_FP_QTANH,
    /* lists: qsum(a...), inner_product(a..., b...) (two halves), polynomial(x, coefficients highest degree first) */
    H2V_FP_QSUM = 40, H2V_FP_INNER_PRODUCT, H2V_FP_POLYNOMIAL,
    /* DistanceInstructions (distance.rs:34-82): (a..., b...) -> distance; also the `distance` argument of
     * nearest_vector / kmeans */
    H2V_DISTANCE_EUCLIDEAN = 60, H2V_DISTANCE_COSINE, H2V_DISTANCE_HAMMING, H2V_DISTANCE_MANHATTAN
};
int h2v_builder_new(uint32_t precision_bits, uint32_t lookup_bits, h2v_builder_t *out);
void h2v_builder_free(h2v_builder_t b);
/* FixedPointChip::quantization / dequantization (fixed_point.rs:104-136) */
int h2v_builder_quantize(h2v_builder_t b, const double *x, size_t n, uint64_t *out_fr);
int h2v_builder_dequantize(h2v_builder_t b, const uint64_t *x_fr, size_t n, double *out);
/* Context::assign_witnesses / load_constant; cell values; the scaffold's `make_public` (mod.rs:376, 400) */
int h2v_builder_assign_witnesses(h2v_builder_t b, const uint64_t *values_fr, size_t n, int64_t *cells_out);
int h2v_builder_load_constant(h2v_builder_t b, const uint64_t value_fr[4], int64_t *cell_out);
int h2v_builder_cell_values(h2v_builder_t b, const int64_t *cells, size_t n, uint64_t *out_fr);
int h2v_builder_make_public(h2v_builder_t b, const int64_t *cells, size_t n);
/* one chip call (H2V_FP_* / H2V_DISTANCE_*) on existing cells */
int h2v_builder_call(h2v_builder_t b, int op, const int64_t *in, size_t n_in, int64_t *out_cell);
/* VectorDBInstructions (/root/reference/src/gadget/vectordb.rs:35-106); vectors: n_vec x dim cells, row-major */
int h2v_builder_nearest_vector(h2v_builder_t b, int distance, const int64_t *query, const int64_t *vectors, size_t n_vec, size_t dim,
                               int64_t *indicator_out /* n_vec */, int64_t *result_out /* dim */);
int h2v_builder_kmeans(h2v_builder_t b, int distance, const int64_t *vectors, size_t n_vec, size_t dim, uint32_t K, uint32_t I,
                       int64_t *centroids_out /* K x dim */, int64_t *indicators_out /* n_vec x K */);
/* PoseidonChip::<F, T, RATE>::new(ctx, r_f, r_p) (examples/query.rs:68; T = 3, RATE = 2 only), one hash
 * (clear / update / squeeze), and merkle_commitment over it */
int h2v_builder_poseidon_new(h2v_builder_t b, uint32_t t, uint32_t rate, uint32_t r_f, uint32_t r_p);
int h2v_builder_poseidon_hash(h2v_builder_t b, const int64_t *in, size_t n, int64_t *out_cell);
int h2v_builder_merkle_commitment(h2v_builder_t b, const int64_t *vectors, size_t n_vec, size_t dim, int64_t *root_out);
/* out: advice cells, lookup cells, distinct constants, public inputs of the trace so far */
int h2v_builder_stats(h2v_builder_t b, uint64_t out[4]);
/* GateThreadBuilder::config(k, Some(minimum_rows)) (mod.rs:383-388): out = num_advice, num_lookup_advice, num_fixed */
int h2v_builder_config(h2v_builder_t b, uint32_t k, uint32_t minimum_rows, uint32_t out[3]);
/* the raw trace (any pointer may be NULL): CANONICAL cell values (4 limbs each), gate selectors, lookup cell offsets */
int h2v_builder_trace(h2v_builder_t b, uint64_t *advice_out, uint8_t *selector_out, int64_t *lookup_out);
/* RangeCircuitBuilder::{mock, keygen, prover} + RangeWithInstanceCircuitBuilder (mod.rs:391-400): the columns of the
 * circuit.  Advice: num_advice gate columns then num_lookup_advice lookup columns; fixed: the lookup table, the
 * constants columns, one selector per gate column; sigma: the permutation over (constants, advice, instance) columns in
 * that order.  Column pointers stay valid until h2v_layout_free. */
int h2v_builder_layout(h2v_builder_t b, uint32_t k, uint32_t minimum_rows, h2v_layout_t *out);
void h2v_layout_free(h2v_layout_t l);
/* out: k, num_advice, num_lookup_advice, num_fixed (constants), public inputs, break points, lookup_bits, minimum_rows */
int h2v_layout_info(h2v_layout_t l, uint32_t out[8]);
int h2v_layout_columns(h2v_layout_t l, int kind /* 0 advice, 1 fixed, 2 sigma */, const uint64_t *const **cols_out, size_t *n_cols);
int h2v_layout_instance(h2v_layout_t l, const uint64_t **out, size_t *n);
/* the pinned break points (configs/<name>.json, mod.rs:272, 285-287) */
int h2v_layout_break_points(h2v_layout_t l, uint32_t *out, size_t cap, size_t *n);

/* ---- Fiat-Shamir transcript, RNG ("next": SURVEY.md 8(f) row 3; host-side, no device needed) ---------------------
 * snark-verifier PoseidonTranscript<G1Affine, NativeLoader, Vec<u8>, T = 5, RATE = 4, R_F = 8, R_P = 60>::new::<0>
 * (scaffold mod.rs:309-310): points are absorbed as (x mod r, y mod r), scalars as themselves; write_* also append the
 * 32-byte encodings below to the proof stream. */
typedef struct h2v_transcript *h2v_transcript_t;
int h2v_transcript_new(h2v_transcript_t *out);
void h2v_transcript_free(h2v_transcript_t t);
int h2v_transcript_common_point(h2v_transcript_t t, const uint64_t affine_pt[8]);
int h2v_transcript_common_scalar(h2v_transcript_t t, const uint64_t scalar[4]);
int h2v_transcript_write_point(h2v_transcript_t t, const uint64_t affine_pt[8]);
int h2v_transcript_write_scalar(h2v_transcript_t t, const uint64_t scalar[4]);
int h2v_transcript_squeeze_challenge(h2v_transcript_t t, uint64_t out[4]);
/* the proof bytes written so far (`finalize()`); out may be NULL to query the length */
int h2v_transcript_bytes(h2v_transcript_t t, uint8_t *out, size_t cap, size_t *len);
/* the Poseidon permutation itself (Grain-LFSR constants, Cauchy MDS; t = 3 or 5) on a Montgomery-form state, in place */
int h2v_poseidon_permutation(uint32_t t, uint32_t r_f, uint32_t r_p, uint64_t *state);
/* variant 0: every round as the Poseidon paper writes it (constants, S-boxes, dense MDS); variant 1: the form the
 * transcript runs (sparse partial rounds, one reduction per matrix row) -- the same permutation, tests compare them */
int h2v_poseidon_permutation_variant(uint32_t t, uint32_t r_f, uint32_t r_p, int variant, uint64_t *state);
/* rand_chacha ChaCha20Rng::from_seed(seed): out[i] = the i-th `Fr::random(&mut rng)` draw (Montgomery form);
 * h2v_chacha20_block = 64 bytes of key stream at a block counter (RFC 7539 block function) */
int h2v_chacha20_fr_random(const uint8_t seed[32], size_t n, uint64_t *out);
int h2v_chacha20_block(const uint8_t seed[32], uint64_t counter, uint8_t out[64]);

/* ---- wire format of commitments and evaluations ("next": SURVEY.md 8(f) row 3; host-side) --------------- */
/* halo2curves 0.3.x G1Affine::to_bytes(): 32 bytes = canonical x little-endian, top bit of byte 31 = parity of
 * canonical y, identity = zeros (recalled, not verified against the crate; halo2curves >= 0.4 uses bit 6) */
int h2v_g1_to_bytes(const uint64_t *affine_pts, size_t n, uint8_t *out);
/* Fr::to_repr(): canonical little-endian 32 bytes per scalar */
int h2v_fr_to_repr(const uint64_t *fr_mont, size_t n, uint8_t *out);

/* ---- device self-tests (used by tests/ to localise failures; not part of the drop-in surface) */
/* out[i] = a[i] (op) b[i] computed by the device field routines; field 0 = Fr, 1 = Fq;
 * op 0 mul, 1 add, 2 sub, 3 inverse by Fermat (b ignored), 4 inverse by binary Euclid (b ignored),
 * 5 the dedicated squaring of a (b ignored), 6 the same on the lazily reduced representative a + m,
 * 7 (Fr only) the NTT's Shoup product: a is ANY 256-bit integer, b a Montgomery twiddle; out = a * from_mont(b) mod r */
int h2v_selftest_field(int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out);
/* out_affine[i] = affine(p[i] + q[i]) through the XYZZ mixed add (mode 0), full add (mode 1) or
 * doubling of p (mode 2); p, q affine */
int h2v_selftest_group(int mode, const uint64_t *p, const uint64_t *q, size_t n, uint64_t *out_affine);
/* synthetic bases with known discrete logs: out[i] = (a*i + b) * G, affine Montgomery (a, b < 2^62);
 * sum_i s_i * out[i] must then equal (sum_i s_i (a i + b) mod r) * G, an algorithm-independent check at any n */
int h2v_synthetic_bases(uint64_t a, uint64_t b, size_t n, uint64_t *out_affine);
/* IMAD.WIDE.U32 (32x32+64 -> 64) issue-rate probe with loop-variant operands: wide multiply-adds per second.
 * This is the integer-pipe roofline denominator (MEASURED_PEAKS.json carries no integer peak). */
int h2v_selftest_imad_peak(double *out_wmac_per_s);
/* which 0: the probe above; 1: a loop of nothing but carry-chained IMAD.WIDE.U32.X rows (the mad.lo.cc / madc.hi.cc
 * pairs the field code is built from) on independent accumulators whose multipliers come from each other -- the
 * roofline denominator that does not depend on any kernel under test */
int h2v_selftest_imad_probe(int which, double *out_wmac_per_s);
/* register-only throughput of the kernels' building blocks, operations per second over the whole GPU:
 * which 0: Fq Montgomery product, one dependent chain per thread; 1: two chains; 2: XYZZ mixed-add chain */
int h2v_selftest_op_rate(int which, double *out_ops_per_s);
/* MSM tuning knobs (tests / tuning; -1 = automatic, the default; also H2V_CHUNK / H2V_TABLE in the environment):
 * `chunk` = sorted entries per accumulate thread; `table` = which of the handle's two window tables a commit uses
 * (0: the window sized for uniform scalars, 1: the smaller window for sparse columns and small calls; automatic =
 * chosen per call from a sampled digit density).  Results do not depend on either. */
int h2v_set_tuning(int chunk, int table);
/* kernels launched by this process so far (for bench.py's gpu_launches) */
uint64_t h2v_launch_count(void);
/* device-side timing of the last commit_batch_dev / transform_dev call, in milliseconds per kernel class:
 * MSM 0 digits 1 scan 2 scatter 3 accumulate 4 finish 5 reduce 6 final; NTT 7 */
int h2v_last_kernel_ms(float out[8]);   /* the calling thread's last call */
/* non-zero digits (= sorted bucket entries = mixed additions msm_accumulate executed) of the calling thread's last
 * h2v_commit_batch_dev: the executed-work figure for the roofline of skewed columns */
uint64_t h2v_last_msm_entries(void);

#ifdef __cplusplus
}
#endif
#endif
