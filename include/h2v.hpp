// h2v.hpp -- header-only C++ mirror of the upstream Rust interface on top of the C ABI (h2v.h).
//
// Same names, argument meaning and error behaviour as halo2-axiom (SURVEY.md 8(a)/(b)):
//   arithmetic.rs            best_multiexp, best_fft
//   poly/kzg/commitment.rs   ParamsKZG::{commit, commit_lagrange}
//   poly/domain.rs           EvaluationDomain::{new, lagrange_to_coeff, coeff_to_extended, extended_to_coeff, ...}
// Upstream panics (assert!) become std::invalid_argument; CUDA failures std::runtime_error (no CPU fallback).
// The reference reaches these through src/scaffold/mod.rs:273 (create_pk) and :296 (gen_snark_shplonk).
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "h2v.h"

namespace h2v_host {

struct Fr { uint64_t l[4]; };          // Montgomery limbs, = halo2curves bn256::Fr
struct G1Affine { uint64_t x[4], y[4]; };
struct G1 { uint64_t x[4], y[4], z[4]; };

inline void check(int rc) {
    if (rc == H2V_OK) return;
    std::string msg = h2v_last_error();
    if (rc == H2V_EINVAL) throw std::invalid_argument(msg);
    throw std::runtime_error(msg);
}
inline void init(int device = 0) { check(h2v_init(&device, 1)); }
inline void init(const std::vector<int> &devices) { check(h2v_init(devices.data(), (int)devices.size())); }

inline G1 best_multiexp(const std::vector<Fr> &coeffs, const std::vector<G1Affine> &bases) {
    if (coeffs.size() != bases.size()) throw std::invalid_argument("assertion failed: coeffs.len() == bases.len()");
    G1 out{};
    check(h2v_best_multiexp(reinterpret_cast<const uint64_t *>(coeffs.data()), reinterpret_cast<const uint64_t *>(bases.data()),
                            coeffs.size(), reinterpret_cast<uint64_t *>(&out)));
    return out;
}
inline void best_fft(std::vector<Fr> &a, const Fr &omega, uint32_t log_n) {
    if (a.size() != (size_t(1) << log_n)) throw std::invalid_argument("assertion failed: a.len() == 1 << log_n");
    check(h2v_best_fft(reinterpret_cast<uint64_t *>(a.data()), omega.l, log_n));
}

// arithmetic.rs eval_polynomial / kate_division, ff BatchInvert, the running product of the permutation argument
inline Fr eval_polynomial(const std::vector<Fr> &poly, const Fr &point) {
    const uint64_t *p[1] = {reinterpret_cast<const uint64_t *>(poly.data())};
    Fr out{};
    check(h2v_eval_polynomial_batch(p, 1, poly.size(), point.l, 1, out.l));
    return out;
}
inline std::vector<Fr> kate_division(const std::vector<Fr> &a, const Fr &b) {
    std::vector<Fr> out(a.empty() ? 0 : a.size() - 1);
    check(h2v_kate_division(reinterpret_cast<const uint64_t *>(a.data()), a.size(), b.l, reinterpret_cast<uint64_t *>(out.data())));
    return out;
}
inline void batch_invert(std::vector<Fr> &a) { check(h2v_batch_invert(reinterpret_cast<uint64_t *>(a.data()), a.size())); }
inline std::vector<Fr> grand_product(const std::vector<Fr> &num, const std::vector<Fr> &den) {
    if (num.size() != den.size()) throw std::invalid_argument("grand_product: length mismatch");
    std::vector<Fr> out(num.size());
    check(h2v_grand_product(reinterpret_cast<const uint64_t *>(num.data()), reinterpret_cast<const uint64_t *>(den.data()), num.size(),
                            reinterpret_cast<uint64_t *>(out.data())));
    return out;
}

class ParamsKZG {
  public:
    ParamsKZG(uint32_t k, const std::vector<G1Affine> &g, const std::vector<G1Affine> &g_lagrange) : k_(k), n_(size_t(1) << k) {
        if ((!g.empty() && g.size() != n_) || (!g_lagrange.empty() && g_lagrange.size() != n_))
            throw std::invalid_argument("ParamsKZG: bases must have 2^k points");
        check(h2v_srs_load(k, g.empty() ? nullptr : reinterpret_cast<const uint64_t *>(g.data()),
                           g_lagrange.empty() ? nullptr : reinterpret_cast<const uint64_t *>(g_lagrange.data()), &h_));
    }
    ~ParamsKZG() { h2v_srs_free(h_); }
    ParamsKZG(const ParamsKZG &) = delete;
    ParamsKZG &operator=(const ParamsKZG &) = delete;
    uint32_t k() const { return k_; }
    size_t n() const { return n_; }
    // commit(&poly, _blind): the blind is ignored by KZG upstream
    G1Affine commit(const std::vector<Fr> &poly) const { return one(H2V_BASIS_MONOMIAL, poly); }
    G1Affine commit_lagrange(const std::vector<Fr> &poly) const { return one(H2V_BASIS_LAGRANGE, poly); }
    std::vector<G1Affine> commit_batch(int basis, const std::vector<const Fr *> &polys, size_t len) const {
        std::vector<G1Affine> out(polys.size());
        check(h2v_commit_batch(h_, basis, reinterpret_cast<const uint64_t *const *>(polys.data()), polys.size(), len,
                               reinterpret_cast<uint64_t *>(out.data())));
        return out;
    }
    h2v_srs_t handle() const { return h_; }

  private:
    G1Affine one(int basis, const std::vector<Fr> &poly) const {
        G1Affine out{};
        check(h2v_commit(h_, basis, reinterpret_cast<const uint64_t *>(poly.data()), poly.size(), reinterpret_cast<uint64_t *>(&out)));
        return out;
    }
    uint32_t k_;
    size_t n_;
    h2v_srs_t h_ = nullptr;
};

class EvaluationDomain {
  public:
    EvaluationDomain(uint32_t j, uint32_t k) : j_(j), k_(k) { check(h2v_domain_new(j, k, &h_)); }
    ~EvaluationDomain() { h2v_domain_free(h_); }
    EvaluationDomain(const EvaluationDomain &) = delete;
    EvaluationDomain &operator=(const EvaluationDomain &) = delete;
    uint32_t k() const { return k_; }
    uint32_t extended_k() const { return h2v_domain_extended_k(h_); }
    size_t extended_len() const { return size_t(1) << extended_k(); }
    uint32_t get_quotient_poly_degree() const { return j_ - 1; }
    Fr get_omega() const { return constant(0); }
    Fr get_omega_inv() const { return constant(1); }
    Fr get_extended_omega() const { return constant(2); }
    Fr constant(int which) const {
        Fr f{};
        check(h2v_domain_constant(h_, which, f.l));
        return f;
    }
    void lagrange_to_coeff(std::vector<Fr> &a) const { need(a.size(), size_t(1) << k_); check(h2v_lagrange_to_coeff(h_, u(a))); }
    void coeff_to_lagrange(std::vector<Fr> &a) const { need(a.size(), size_t(1) << k_); check(h2v_coeff_to_lagrange(h_, u(a))); }
    std::vector<Fr> coeff_to_extended(const std::vector<Fr> &a) const {
        need(a.size(), size_t(1) << k_);
        std::vector<Fr> out(extended_len());
        check(h2v_coeff_to_extended(h_, reinterpret_cast<const uint64_t *>(a.data()), u(out)));
        return out;
    }
    std::vector<Fr> extended_to_coeff(const std::vector<Fr> &a) const {
        need(a.size(), extended_len());
        std::vector<Fr> out((size_t(1) << k_) * (j_ - 1));
        check(h2v_extended_to_coeff(h_, reinterpret_cast<const uint64_t *>(a.data()), u(out)));
        return out;
    }
    void divide_by_vanishing_poly(std::vector<Fr> &a) const { need(a.size(), extended_len()); check(h2v_divide_by_vanishing_poly(h_, u(a))); }
    // poly/domain.rs scalar / index helpers (host-side)
    Fr rotate_omega(const Fr &value, int32_t rotation) const {
        Fr f{};
        check(h2v_domain_rotate_omega(h_, value.l, rotation, f.l));
        return f;
    }
    std::vector<Fr> rotate_extended(const std::vector<Fr> &poly, int32_t rotation) const {
        need(poly.size(), extended_len());
        std::vector<Fr> out(poly.size());
        check(h2v_domain_rotate_extended(h_, reinterpret_cast<const uint64_t *>(poly.data()), rotation, u(out)));
        return out;
    }
    // l_i_range(x, xn, lo..hi): l_i(x) for lo <= i < hi
    std::vector<Fr> l_i_range(const Fr &x, const Fr &xn, int32_t lo, int32_t hi) const {
        std::vector<Fr> out(hi > lo ? size_t(hi - lo) : 0);
        check(h2v_domain_l_i_range(h_, x.l, xn.l, lo, hi, u(out)));
        return out;
    }
    std::vector<Fr> empty_coeff() const { return fill(0, nullptr); }
    std::vector<Fr> empty_lagrange() const { return fill(1, nullptr); }
    std::vector<Fr> empty_extended() const { return fill(2, nullptr); }
    std::vector<Fr> constant_lagrange(const Fr &scalar) const { return fill(1, &scalar); }
    std::vector<Fr> constant_extended(const Fr &scalar) const { return fill(2, &scalar); }
    h2v_domain_t handle() const { return h_; }

    // evaluate_h's row loops on device-resident extended columns (plonk/evaluation.rs [UPSTREAM]); pointers are
    // device pointers from h2v_dev_alloc, columns `stride` Fr elements apart; h <- h * y + term, in upstream's order
    void quotient_gates(void *d_h, const Fr &y, size_t n_gates, const void *d_q, size_t q_stride, const void *d_a, size_t a_stride) const {
        check(h2v_quotient_gates_dev(h_, d_h, y.l, n_gates, d_q, q_stride, d_a, a_stride));
    }
    void quotient_permutation(void *d_h, const Fr &y, const Fr &beta, const Fr &gamma, size_t n_cols, size_t chunk_len, const void *d_cols,
                              size_t cols_stride, const void *d_sigma, size_t sigma_stride, const void *d_z, size_t z_stride,
                              const void *d_l0, const void *d_l_last, const void *d_l_active, uint32_t blinding_factors) const {
        check(h2v_quotient_permutation_dev(h_, d_h, y.l, beta.l, gamma.l, n_cols, chunk_len, d_cols, cols_stride, d_sigma, sigma_stride,
                                           d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors));
    }
    // the same fold over the permutation sets [set_begin, set_end) only (extended columns streamed in slices, k = 20)
    void quotient_permutation_range(void *d_h, const Fr &y, const Fr &beta, const Fr &gamma, size_t n_cols, size_t chunk_len, size_t set_begin,
                                    size_t set_end, bool with_head, const void *const *d_col_ptrs, const void *const *d_sigma_ptrs,
                                    const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last, const void *d_l_active,
                                    uint32_t blinding_factors) const {
        check(h2v_quotient_permutation_range_ptrs_dev(h_, d_h, y.l, beta.l, gamma.l, n_cols, chunk_len, set_begin, set_end, with_head ? 1 : 0,
                                                      d_col_ptrs, d_sigma_ptrs, d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors));
    }
    void quotient_lookup(void *d_h, const Fr &y, const Fr &beta, const Fr &gamma, const void *d_input, const void *d_table,
                         const void *d_perm_input, const void *d_perm_table, const void *d_z, const void *d_l0, const void *d_l_last,
                         const void *d_l_active) const {
        check(h2v_quotient_lookup_dev(h_, d_h, y.l, beta.l, gamma.l, d_input, d_table, d_perm_input, d_perm_table, d_z, d_l0, d_l_last,
                                      d_l_active));
    }

  private:
    std::vector<Fr> fill(int basis, const Fr *scalar) const {
        std::vector<Fr> out(basis == 2 ? extended_len() : size_t(1) << k_);
        check(h2v_domain_fill(h_, basis, scalar ? scalar->l : nullptr, u(out)));
        return out;
    }
    static uint64_t *u(std::vector<Fr> &v) { return reinterpret_cast<uint64_t *>(v.data()); }
    static void need(size_t got, size_t want) {
        if (got != want) throw std::invalid_argument("assertion failed: polynomial length does not match the domain");
    }
    uint32_t j_, k_;
    h2v_domain_t h_ = nullptr;
};

// plonk/lookup/prover.rs permute_expression_pair [UPSTREAM]: (permuted_input, permuted_table) of the usable rows;
// throws std::invalid_argument when an input value is missing from the table (upstream: ConstraintSystemFailure)
inline std::pair<std::vector<Fr>, std::vector<Fr>> permute_expression_pair(const std::vector<Fr> &input, const std::vector<Fr> &table) {
    if (input.size() != table.size()) throw std::invalid_argument("input and table must have the same number of usable rows");
    std::vector<Fr> a(input.size()), s(input.size());
    check(h2v_permute_expression_pair(reinterpret_cast<const uint64_t *>(input.data()), reinterpret_cast<const uint64_t *>(table.data()),
                                      input.size(), reinterpret_cast<uint64_t *>(a.data()), reinterpret_cast<uint64_t *>(s.data())));
    return {std::move(a), std::move(s)};
}

// snark-verifier PoseidonTranscript<G1Affine, NativeLoader, Vec<u8>, 5, 4, 8, 60>::new::<0> (scaffold mod.rs:309-310), host-side
class PoseidonTranscript {
  public:
    PoseidonTranscript() { check(h2v_transcript_new(&h_)); }
    ~PoseidonTranscript() { h2v_transcript_free(h_); }
    PoseidonTranscript(const PoseidonTranscript &) = delete;
    PoseidonTranscript &operator=(const PoseidonTranscript &) = delete;
    void common_point(const G1Affine &p) { check(h2v_transcript_common_point(h_, reinterpret_cast<const uint64_t *>(&p))); }
    void common_scalar(const Fr &s) { check(h2v_transcript_common_scalar(h_, s.l)); }
    void write_point(const G1Affine &p) { check(h2v_transcript_write_point(h_, reinterpret_cast<const uint64_t *>(&p))); }
    void write_scalar(const Fr &s) { check(h2v_transcript_write_scalar(h_, s.l)); }
    Fr squeeze_challenge() {
        Fr f{};
        check(h2v_transcript_squeeze_challenge(h_, f.l));
        return f;
    }
    std::vector<uint8_t> finalize() const {
        size_t len = 0;
        check(h2v_transcript_bytes(h_, nullptr, 0, &len));
        std::vector<uint8_t> out(len);
        if (len) check(h2v_transcript_bytes(h_, out.data(), len, &len));
        return out;
    }

  private:
    h2v_transcript_t h_ = nullptr;
};

// halo2 MockProver::run(k, circuit, instances) on the device (h2v_mock_prover): the first max_failures failures in the order
// gates, lookups, permutation, and how many there are in all
struct MockProver {
    std::vector<h2v_mock_failure_t> failures;
    uint64_t n_failures = 0;

    static MockProver run(const h2v_circuit_t &cs, const std::vector<const Fr *> &fixed, const std::vector<const Fr *> &sigma,
                          const std::vector<const Fr *> &advice, const std::vector<std::vector<Fr>> &instances, size_t max_failures = 64) {
        if (fixed.size() != cs.n_fixed || sigma.size() != cs.n_perm || advice.size() != cs.n_advice || instances.size() != cs.n_instance)
            throw std::invalid_argument("MockProver: column count does not match the constraint system");
        std::vector<const uint64_t *> ip;
        std::vector<uint32_t> il;
        for (const auto &c : instances) {
            ip.push_back(reinterpret_cast<const uint64_t *>(c.data()));
            il.push_back((uint32_t)c.size());
        }
        MockProver m;
        m.failures.resize(max_failures);
        check(h2v_mock_prover(&cs, reinterpret_cast<const uint64_t *const *>(fixed.data()), reinterpret_cast<const uint64_t *const *>(sigma.data()),
                              reinterpret_cast<const uint64_t *const *>(advice.data()), ip.data(), il.data(), m.failures.data(), max_failures,
                              &m.n_failures));
        m.failures.resize((size_t)std::min<uint64_t>(max_failures, m.n_failures));
        return m;
    }
    // MockProver::assert_satisfied: throws std::logic_error naming the first failures
    void assert_satisfied() const {
        if (!n_failures) return;
        static const char *kinds[] = {"?", "gate", "gate_unusable", "lookup", "sigma_not_delta_omega", "sigma_not_permutation", "copy_unusable", "copy"};
        std::string msg = std::to_string(n_failures) + " constraint(s) not satisfied";
        for (const auto &f : failures)
            msg += "\n  " + std::string(kinds[f.kind < 8 ? f.kind : 0]) + ": column " + std::to_string(f.column) + " row " + std::to_string(f.row) +
                   " (other: column " + std::to_string(f.other_column) + " row " + std::to_string(f.other_row) + ")";
        throw std::logic_error(msg);
    }
};

class WitnessProgram;

// halo2 ProvingKey for a halo2-base-shaped constraint system + create_proof (plonk/prover.rs), resident on the device
class ProvingKey {
  public:
    ProvingKey(const ParamsKZG &params, const h2v_circuit_t &cs, const std::vector<const Fr *> &fixed, const std::vector<const Fr *> &sigma,
               const Fr &vk_transcript_repr) {
        check(h2v_pk_load(params.handle(), &cs, reinterpret_cast<const uint64_t *const *>(fixed.data()),
                          reinterpret_cast<const uint64_t *const *>(sigma.data()), vk_transcript_repr.l, &h_));
    }
    ~ProvingKey() { h2v_pk_free(h_); }
    ProvingKey(const ProvingKey &) = delete;
    ProvingKey &operator=(const ProvingKey &) = delete;
    // create_proof(params, pk, &[circuit], &[instances], ChaCha20Rng::from_seed(seed), transcript) -> transcript.finalize()
    std::vector<uint8_t> create_proof(const std::vector<const Fr *> &advice, const std::vector<std::vector<Fr>> &instances,
                                      const std::array<uint8_t, 32> &rng_seed) const {
        std::vector<const uint64_t *> ip;
        std::vector<uint32_t> il;
        for (const auto &c : instances) {
            ip.push_back(reinterpret_cast<const uint64_t *>(c.data()));
            il.push_back((uint32_t)c.size());
        }
        std::vector<uint8_t> out(h2v_proof_size(h_));
        size_t len = 0;
        check(h2v_create_proof(h_, reinterpret_cast<const uint64_t *const *>(advice.data()), ip.data(), il.data(), rng_seed.data(), out.data(),
                               out.size(), &len));
        out.resize(len);
        return out;
    }
    // proof p = create_proof(advice[p], instances[p], rng_seeds[p]), the proofs run in groups (h2v_create_proofs)
    std::vector<std::vector<uint8_t>> create_proofs(const std::vector<std::vector<const Fr *>> &advice,
                                                    const std::vector<std::vector<std::vector<Fr>>> &instances,
                                                    const std::vector<std::array<uint8_t, 32>> &rng_seeds) const {
        const size_t B = advice.size();
        if (instances.size() != B || rng_seeds.size() != B) throw std::invalid_argument("create_proofs: list lengths differ");
        std::vector<std::vector<const uint64_t *>> ip(B);
        std::vector<std::vector<uint32_t>> il(B);
        std::vector<const uint64_t *const *> ap(B), ipp(B);
        std::vector<const uint32_t *> ilp(B);
        std::vector<uint8_t> seeds(32 * B);
        for (size_t p = 0; p < B; ++p) {
            for (const auto &c : instances[p]) {
                ip[p].push_back(reinterpret_cast<const uint64_t *>(c.data()));
                il[p].push_back((uint32_t)c.size());
            }
            ap[p] = reinterpret_cast<const uint64_t *const *>(advice[p].data());
            ipp[p] = ip[p].data();
            ilp[p] = il[p].data();
            std::copy(rng_seeds[p].begin(), rng_seeds[p].end(), seeds.begin() + 32 * p);
        }
        const size_t size = h2v_proof_size(h_);
        std::vector<uint8_t> flat(B * size);
        check(h2v_create_proofs(h_, B, ap.data(), ipp.data(), ilp.data(), seeds.data(), flat.data(), size));
        std::vector<std::vector<uint8_t>> out(B);
        for (size_t p = 0; p < B; ++p) out[p].assign(flat.begin() + p * size, flat.begin() + (p + 1) * size);
        return out;
    }
    // MockProver::run on this key's circuit for each witness: result w = MockProver::run(cs, fixed, sigma, advice[w],
    // instances[w], max_failures) with the key's cs, fixed and sigma; one call for the whole batch (h2v_pk_mock_prover)
    std::vector<MockProver> mock_prover(const std::vector<std::vector<const Fr *>> &advice, const std::vector<std::vector<std::vector<Fr>>> &instances,
                                        size_t max_failures = 64) const {
        const size_t B = advice.size();
        if (instances.size() != B) throw std::invalid_argument("mock_prover: list lengths differ");
        std::vector<std::vector<const uint64_t *>> ip(B);
        std::vector<std::vector<uint32_t>> il(B);
        std::vector<const uint64_t *const *> ap(B), ipp(B);
        std::vector<const uint32_t *> ilp(B);
        for (size_t w = 0; w < B; ++w) {
            for (const auto &c : instances[w]) {
                ip[w].push_back(reinterpret_cast<const uint64_t *>(c.data()));
                il[w].push_back((uint32_t)c.size());
            }
            ap[w] = reinterpret_cast<const uint64_t *const *>(advice[w].data());
            ipp[w] = ip[w].data();
            ilp[w] = il[w].data();
        }
        std::vector<h2v_mock_failure_t> flat(B * max_failures);
        std::vector<uint64_t> totals(B);
        check(h2v_pk_mock_prover(h_, B, ap.data(), ipp.data(), ilp.data(), flat.data(), max_failures, totals.data()));
        std::vector<MockProver> out(B);
        for (size_t w = 0; w < B; ++w) {
            out[w].n_failures = totals[w];
            out[w].failures.assign(flat.begin() + w * max_failures, flat.begin() + w * max_failures + (size_t)std::min<uint64_t>(max_failures, totals[w]));
        }
        return out;
    }
    // create_proofs on the columns program.generate gives for inputs (n_proofs x n_inputs values), generated in this key's
    // workspace without crossing to the host (h2v_create_proofs_from_inputs); instances: n_proofs x program.n_instances()
    std::vector<std::vector<uint8_t>> create_proofs_from_inputs(const WitnessProgram &program, size_t n_proofs, const std::vector<Fr> &inputs,
                                                                const std::vector<std::array<uint8_t, 32>> &rng_seeds, std::vector<Fr> &instances) const;
    // mock_prover on the same generated columns (h2v_pk_mock_prover_from_inputs)
    std::vector<MockProver> mock_prover_from_inputs(const WitnessProgram &program, size_t n_witnesses, const std::vector<Fr> &inputs,
                                                    size_t max_failures = 64) const;

  private:
    h2v_pk_t h_ = nullptr;
};

// A recorded circuit replayed for many inputs on the GPU (h2v_witness_program_new / h2v_witness_generate).  The builder
// must come from h2v_builder_new_recording; it may be freed once the program exists.
class WitnessProgram {
  public:
    WitnessProgram(h2v_builder_t recording, uint32_t k, uint32_t minimum_rows = 9) {
        check(h2v_witness_program_new(recording, k, minimum_rows, &h_));
        check(h2v_witness_program_info(h_, info_));
    }
    ~WitnessProgram() { h2v_witness_program_free(h_); }
    WitnessProgram(const WitnessProgram &) = delete;
    WitnessProgram &operator=(const WitnessProgram &) = delete;
    size_t n_inputs() const { return (size_t)info_[0]; }
    size_t n_advice() const { return (size_t)info_[4]; }
    size_t n_instances() const { return (size_t)info_[5]; }
    h2v_witness_program_t handle() const { return h_; }
    // inputs: n_witnesses x n_inputs values -> advice (n_witnesses x n_advice x 2^k) and instances (n_witnesses x n_instances)
    void generate(size_t n_witnesses, const std::vector<Fr> &inputs, std::vector<Fr> &advice, std::vector<Fr> &instances) const {
        if (inputs.size() != n_witnesses * n_inputs()) throw std::invalid_argument("witness_generate: inputs.size() != n_witnesses * n_inputs");
        advice.resize(n_witnesses * n_advice() * ((size_t)1 << info_[6]));
        instances.resize(n_witnesses * n_instances());
        check(h2v_witness_generate(h_, n_witnesses, n_inputs(), inputs.empty() ? nullptr : &inputs[0].l[0], &advice[0].l[0],
                                   instances.empty() ? nullptr : &instances[0].l[0]));
    }

  private:
    h2v_witness_program_t h_ = nullptr;
    uint64_t info_[8] = {};
};

inline std::vector<std::vector<uint8_t>> ProvingKey::create_proofs_from_inputs(const WitnessProgram &program, size_t n_proofs,
                                                                               const std::vector<Fr> &inputs,
                                                                               const std::vector<std::array<uint8_t, 32>> &rng_seeds,
                                                                               std::vector<Fr> &instances) const {
    if (inputs.size() != n_proofs * program.n_inputs() || rng_seeds.size() != n_proofs)
        throw std::invalid_argument("create_proofs_from_inputs: inputs.size() != n_proofs * n_inputs or rng_seeds.size() != n_proofs");
    std::vector<uint8_t> seeds(32 * n_proofs);
    for (size_t p = 0; p < n_proofs; ++p) std::copy(rng_seeds[p].begin(), rng_seeds[p].end(), seeds.begin() + 32 * p);
    instances.resize(n_proofs * program.n_instances());
    const size_t size = h2v_proof_size(h_);
    std::vector<uint8_t> flat(n_proofs * size);
    check(h2v_create_proofs_from_inputs(h_, program.handle(), n_proofs, program.n_inputs(), inputs.empty() ? nullptr : &inputs[0].l[0],
                                        seeds.data(), flat.data(), size, instances.empty() ? nullptr : &instances[0].l[0]));
    std::vector<std::vector<uint8_t>> out(n_proofs);
    for (size_t p = 0; p < n_proofs; ++p) out[p].assign(flat.begin() + p * size, flat.begin() + (p + 1) * size);
    return out;
}
inline std::vector<MockProver> ProvingKey::mock_prover_from_inputs(const WitnessProgram &program, size_t n_witnesses, const std::vector<Fr> &inputs,
                                                                   size_t max_failures) const {
    if (inputs.size() != n_witnesses * program.n_inputs()) throw std::invalid_argument("mock_prover_from_inputs: inputs.size() != n_witnesses * n_inputs");
    std::vector<h2v_mock_failure_t> flat(n_witnesses * max_failures);
    std::vector<uint64_t> totals(n_witnesses);
    check(h2v_pk_mock_prover_from_inputs(h_, program.handle(), n_witnesses, program.n_inputs(), inputs.empty() ? nullptr : &inputs[0].l[0],
                                         flat.data(), max_failures, totals.data()));
    std::vector<MockProver> out(n_witnesses);
    for (size_t w = 0; w < n_witnesses; ++w) {
        out[w].n_failures = totals[w];
        out[w].failures.assign(flat.begin() + w * max_failures, flat.begin() + w * max_failures + (size_t)std::min<uint64_t>(max_failures, totals[w]));
    }
    return out;
}

}  // namespace h2v_host
