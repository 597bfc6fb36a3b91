// prover.cu -- create_proof over the library's kernels: one Halo2-KZG (SHPLONK) proof of one halo2-base-shaped
// circuit, every column resident in HBM from upload to the last commitment ("next" rows 2-3 of SURVEY.md 8(f)).
//
// Restates the control flow of [UPSTREAM] halo2-axiom (PSE v2023_02_02 lineage, /root/reference/Cargo.toml:19-22)
//   plonk/prover.rs `create_proof`, plonk/{lookup,permutation,vanishing}/prover.rs, plonk/evaluation.rs `evaluate_h`,
//   poly/kzg/multiopen/shplonk/prover.rs `ProverSHPLONK::create_proof` + shplonk.rs `construct_intermediate_sets`
// as it is reached from /root/reference/src/scaffold/mod.rs:296 (`gen_snark_shplonk`) with the transcript of
// mod.rs:309-310.  The host code below only sequences: Fiat-Shamir challenges, the seeded RNG draws in upstream's
// order, the point sets of the multi-open argument.  All arithmetic on columns is done by kernels -- the MSM / NTT /
// quotient / grand-product / permutation kernels behind the C ABI `_dev` entry points (h2v.cu) and the small
// column kernels in this file.
//
// Constraint-system shape (what halo2-base's FlexGateConfig / RangeConfig produce, [UPSTREAM] gates/{flex_gate,range}.rs):
//   gate j      q_j(X) * (a_j(X) + a_j(wX) a_j(w^2 X) - a_j(w^3 X))       one per "basic gate" advice column
//   lookup l    single-expression input (an advice column) in a single-expression table (a fixed column)
//   permutation any list of advice / fixed / instance columns
// One advice phase, no challenges inside the witness (halo2-base's default), QUERY_INSTANCE = false (KZG).
// What is recalled rather than verified against upstream text is listed in DESIGN.md ("recalled conventions").
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <vector>

#include "h2v.h"
#include "internal.hpp"
#include "ec.cuh"
#include "fr_host.hpp"
#include "chacha.hpp"
#include "poseidon.hpp"
#include "g2_host.hpp"

using namespace h2v;

namespace h2v {
const PoseidonSpec<5> &poseidon_transcript_spec() {
    static const PoseidonSpec<5> spec = poseidon_make_spec<5>(8, 60);
    return spec;
}
}  // namespace h2v

namespace {

typedef FrP Fr;

// ------------------------------------------------------------------ column kernels
__device__ __forceinline__ fe ld(const fe *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = q[0], b = q[1];
    fe r;
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    return r;
}
__device__ __forceinline__ void st(fe *p, const fe &x) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    q[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
}

// permutation argument, plonk/permutation/prover.rs `Argument::commit`: for set s (grid.y) and row i
//   den[s][i] = prod_{c in set} (v_c[i] + beta sigma_c[i] + gamma),  num[s][i] = prod (v_c[i] + beta delta^c w^i + gamma)
struct PermArgs {
    const fe *const *cols;      // n_cols Lagrange columns in permutation order
    const fe *const *sigma;     // their sigma polynomials, Lagrange
    const fe *omega_pows;       // w^i
    const fe *delta_start;      // per set: delta^(s * chunk)
    fe beta, gamma, delta;
    uint32_t n_cols, chunk, n;
};
__global__ void __launch_bounds__(256) perm_numden_kernel(PermArgs a, fe *num, fe *den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y;
    if (i >= a.n) return;
    const uint32_t c0 = s * a.chunk, c1 = min(c0 + a.chunk, a.n_cols);
    fe cur = fe_mul<Fr>(fe_mul<Fr>(a.beta, ld(a.omega_pows + i)), ld(a.delta_start + s));
    fe nu = fe_one<Fr>(), de = fe_one<Fr>();
    for (uint32_t c = c0; c < c1; ++c) {
        const fe v = fe_add<Fr>(ld(a.cols[c] + i), a.gamma);
        de = fe_mul<Fr>(de, fe_add<Fr>(v, fe_mul<Fr>(a.beta, ld(a.sigma[c] + i))));
        nu = fe_mul<Fr>(nu, fe_add<Fr>(v, cur));
        cur = fe_mul<Fr>(cur, a.delta);
    }
    st(num + (size_t)s * a.n + i, nu);
    st(den + (size_t)s * a.n + i, de);
}
// lookup argument, plonk/lookup/prover.rs `Permuted::commit_product`: for lookup l (grid.y) and row i
//   den = (a'[i] + beta)(s'[i] + gamma),  num = (a[i] + beta)(t[i] + gamma)
__global__ void __launch_bounds__(256) lookup_numden_kernel(const fe *const *inputs, const fe *const *tables, const fe *perm_in,
                                                            const fe *perm_tab, fe beta, fe gamma, uint32_t n, fe *num, fe *den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y;
    if (i >= n) return;
    const size_t o = (size_t)l * n + i;
    st(num + o, fe_mul<Fr>(fe_add<Fr>(ld(inputs[l] + i), beta), fe_add<Fr>(ld(tables[l] + i), gamma)));
    st(den + o, fe_mul<Fr>(fe_add<Fr>(ld(perm_in + o), beta), fe_add<Fr>(ld(perm_tab + o), gamma)));
}
// cols[c][i] *= scalars[c]   (n_cols contiguous columns of n)
__global__ void __launch_bounds__(256) scale_cols_kernel(fe *cols, uint32_t n, const fe *scalars) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe *p = cols + (size_t)blockIdx.y * n + i;
    st(p, fe_mul<Fr>(ld(p), ld(scalars + blockIdx.y)));
}
// out[i] = sum_j coef[j] * cols[j][i]
__global__ void __launch_bounds__(256) lincomb_kernel(const fe *const *cols, const fe *coef, uint32_t n_cols, uint32_t n, fe *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe acc = fe_zero();
    for (uint32_t j = 0; j < n_cols; ++j) acc = fe_add<Fr>(acc, fe_mul<Fr>(ld(cols[j] + i), ld(coef + j)));
    st(out + i, acc);
}
// a[i] -= low[i], i < cnt   (subtracting a low-degree polynomial)
__global__ void sub_low_kernel(fe *a, const fe *low, uint32_t cnt) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) st(a + i, fe_sub<Fr>(ld(a + i), ld(low + i)));
}
// arithmetic.rs eval_polynomial for a list of (polynomial, point) pairs: one CTA per pair, Horner over 256 slices
struct EvalPair {
    const fe *poly;
    uint32_t point;
};
__global__ void __launch_bounds__(256) eval_pairs_kernel(const EvalPair *pairs, const fe *points, uint32_t len, fe *out) {
    __shared__ fe sm8[8];
    const EvalPair pr = pairs[blockIdx.x];
    const fe x = ld(points + pr.point);
    const uint32_t chunk = (len + 255) / 256;
    const uint32_t lo = min(threadIdx.x * chunk, len), hi = min(lo + chunk, len);
    fe v = fe_zero();
    for (uint32_t i = hi; i-- > lo;) v = fe_add<Fr>(fe_mul<Fr>(v, x), ld(pr.poly + i));
    v = fe_mul<Fr>(v, fe_pow_small<Fr>(fe_pow_small<Fr>(x, chunk), threadIdx.x));
#pragma unroll 1
    for (int o = 16; o >= 1; o >>= 1) {
        fe t;
#pragma unroll
        for (int k = 0; k < 8; ++k) t.v[k] = __shfl_down_sync(0xffffffffu, v.v[k], o);
        v = fe_add<Fr>(v, t);
    }
    if ((threadIdx.x & 31) == 0) sm8[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        fe s = sm8[0];
        for (int w = 1; w < 8; ++w) s = fe_add<Fr>(s, sm8[w]);
        st(out + blockIdx.x, s);
    }
}

// out[i] = the `Fr::random` draw that consumes key-stream block counter0 + i (chacha.hpp): the ChaCha20 block function and
// the reduction of its 512-bit little-endian value mod r, one thread per draw (the vanishing argument's random
// polynomial is n consecutive draws)
__device__ __forceinline__ uint32_t rotl32(uint32_t v, int n) { return (v << n) | (v >> (32 - n)); }
#define H2V_QR(a, b, c, d)                 \
    a += b; d = rotl32(d ^ a, 16);         \
    c += d; b = rotl32(b ^ c, 12);         \
    a += b; d = rotl32(d ^ a, 8);          \
    c += d; b = rotl32(b ^ c, 7);
struct ChaChaKey {
    uint32_t k[8];
};
__device__ __forceinline__ fe canon_below_2_256(fe v) {      // v < 2^256 < 6r  ->  v mod r
    // subtract 4r, 2r, r when possible
#pragma unroll
    for (int sh = 2; sh >= 0; --sh) {
        uint32_t m[8], d[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint64_t w = ((uint64_t)Fr::m(i) << sh) | (i ? ((uint64_t)Fr::m(i - 1) >> (32 - sh)) : 0);
            m[i] = (uint32_t)w;
        }
        const uint32_t bw = raw_sub(d, v.v, m);
#pragma unroll
        for (int i = 0; i < 8; ++i) v.v[i] = bw ? v.v[i] : d[i];
    }
    return v;
}
__global__ void __launch_bounds__(256) chacha_fr_kernel(ChaChaKey key, uint64_t counter0, uint32_t n, fe *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t ctr = counter0 + i;
    uint32_t x0 = 0x61707865u, x1 = 0x3320646eu, x2 = 0x79622d32u, x3 = 0x6b206574u;
    uint32_t x4 = key.k[0], x5 = key.k[1], x6 = key.k[2], x7 = key.k[3], x8 = key.k[4], x9 = key.k[5], x10 = key.k[6], x11 = key.k[7];
    uint32_t x12 = (uint32_t)ctr, x13 = (uint32_t)(ctr >> 32), x14 = 0, x15 = 0;
    const uint32_t i12 = x12, i13 = x13;
#pragma unroll 1
    for (int r = 0; r < 10; ++r) {
        H2V_QR(x0, x4, x8, x12) H2V_QR(x1, x5, x9, x13) H2V_QR(x2, x6, x10, x14) H2V_QR(x3, x7, x11, x15)
        H2V_QR(x0, x5, x10, x15) H2V_QR(x1, x6, x11, x12) H2V_QR(x2, x7, x8, x13) H2V_QR(x3, x4, x9, x14)
    }
    fe lo, hi;
    lo.v[0] = x0 + 0x61707865u; lo.v[1] = x1 + 0x3320646eu; lo.v[2] = x2 + 0x79622d32u; lo.v[3] = x3 + 0x6b206574u;
    lo.v[4] = x4 + key.k[0]; lo.v[5] = x5 + key.k[1]; lo.v[6] = x6 + key.k[2]; lo.v[7] = x7 + key.k[3];
    hi.v[0] = x8 + key.k[4]; hi.v[1] = x9 + key.k[5]; hi.v[2] = x10 + key.k[6]; hi.v[3] = x11 + key.k[7];
    hi.v[4] = x12 + i12; hi.v[5] = x13 + i13; hi.v[6] = x14; hi.v[7] = x15;
    // (lo + hi 2^256) mod r in Montgomery form: to_mont(lo) + to_mont(to_mont(hi))
    const fe a = fe_to_mont<Fr>(canon_below_2_256(lo)), b = fe_to_mont<Fr>(fe_to_mont<Fr>(canon_below_2_256(hi)));
    st(out + i, fe_add<Fr>(a, b));
}

// ------------------------------------------------------------------ small host helpers
inline const uint64_t *u64(const Fr64 &a) { return a.l; }

// Lagrange basis over the points xs: basis[j] = coefficients of prod_{k != j} (X - x_k) / prod_{k != j} (x_j - x_k).
// One rotation set shares its points between hundreds of polynomials, so the basis (and its m inversions) is built once
// per set; the polynomial through (xs[i], ys[i]) (arithmetic.rs lagrange_interpolate) is then sum_j ys[j] basis[j].
std::vector<std::vector<Fr64>> lagrange_basis(const std::vector<Fr64> &xs) {
    const size_t m = xs.size();
    std::vector<std::vector<Fr64>> basis(m);
    for (size_t j = 0; j < m; ++j) {
        std::vector<Fr64> num(1, frh::ONE);
        Fr64 den = frh::ONE;
        for (size_t k = 0; k < m; ++k) {
            if (k == j) continue;
            std::vector<Fr64> nx(num.size() + 1, frh::zero());
            for (size_t t = 0; t < num.size(); ++t) {
                nx[t + 1] = frh::add(nx[t + 1], num[t]);
                nx[t] = frh::sub(nx[t], frh::mul(num[t], xs[k]));
            }
            num.swap(nx);
            den = frh::mul(den, frh::sub(xs[j], xs[k]));
        }
        const Fr64 di = m == 1 ? frh::ONE : frh::inv(den);
        for (Fr64 &c : num) c = frh::mul(c, di);
        basis[j].swap(num);
    }
    return basis;
}
std::vector<Fr64> lagrange_interpolate(const std::vector<std::vector<Fr64>> &basis, const std::vector<Fr64> &ys) {
    const size_t m = basis.size();
    std::vector<Fr64> out(m, frh::zero());
    for (size_t j = 0; j < m; ++j)
        for (size_t t = 0; t < m; ++t) out[t] = frh::add(out[t], frh::mul(basis[j][t], ys[j]));
    return out;
}
Fr64 eval_small(const std::vector<Fr64> &poly, const Fr64 &x) {
    Fr64 acc = frh::zero();
    for (size_t i = poly.size(); i-- > 0;) acc = frh::add(frh::mul(acc, x), poly[i]);
    return acc;
}

}  // namespace

// ================================================================== proving key handle
struct h2v_pk {
    h2v_srs_t srs = nullptr;
    h2v_domain_t dom = nullptr;
    uint32_t k = 0, degree = 0, bf = 0, n_advice = 0, n_fixed = 0, n_instance = 0;
    std::vector<uint32_t> gate_advice, gate_selector, lookup_input, lookup_table, perm_index, aq_col, fq_col;
    std::vector<uint8_t> perm_kind;
    std::vector<int32_t> aq_rot, fq_rot;
    size_t n = 0, ne = 0;
    uint32_t u = 0, chunk = 0, n_sets = 0;
    Fr64 vk_repr, omega, omega_inv, delta;
    DevBuf fixed_L, fixed_C, fixed_E, sigma_L, sigma_C, sigma_E, lrows_E, omega_pows;
    // per-proof workspace, kept between proofs
    DevBuf adv_L, adv_C, adv_E, inst_L, inst_C, inst_E, pa_L, ps_L, pa_C, ps_C, pa_E, ps_E, z_L, z_C, z_E, zl_L, zl_C, zl_E;
    DevBuf num, den, tails, ptrs, scal, pts, rnd_C, hq, hx_pieces, evals, pairs, sh_S, sh_A, sh_B, sh_h, commits;
    // k = 20-sized keys: the extended-coset forms of the fixed / sigma / advice columns (4n each) are not kept -- the
    // quotient step rebuilds them from the coefficient forms in slices of `scr_cols` columns of `scr_E`
    bool stream_ext = false;
    size_t scr_cols = 0;
    DevBuf scr_E;
    // ... and what is left of the device's memory after the first proof's buffers exist keeps the extended forms of the first
    // `cached_sigma` sigma polynomials (they belong to the key: every later proof skips their coeff_to_extended)
    DevBuf ext_cache;
    size_t cached_sigma = 0;
    bool cache_tried = false;
    cudaStream_t st = nullptr;
    int dev = 0;                 // the proof runs on the primary device (columns and key resident there)
    std::mutex mu;
    double last_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // wall-clock per phase of the last create_proof
};

namespace {

int sync(h2v_pk *pk) {
    H2V_CU(cudaStreamSynchronize(pk->st));
    return H2V_OK;
}
// upload a host array of device pointers / scalars into a (reused) device buffer at byte offset `off`
int upload(h2v_pk *pk, DevBuf &b, size_t off, const void *src, size_t bytes) {
    H2V_CU(cudaMemcpyAsync((char *)b.p + off, src, bytes, cudaMemcpyHostToDevice, pk->st));
    H2V_CU(cudaStreamSynchronize(pk->st));      // the host staging vectors are short-lived
    return H2V_OK;
}
// rows [row0, row0 + rows) of `n_cols` contiguous columns of n <- tails (n_cols x rows, host)
int write_rows(h2v_pk *pk, fe *cols, size_t n, size_t row0, size_t rows, size_t n_cols, const std::vector<Fr64> &tails) {
    if (!rows || !n_cols) return H2V_OK;
    H2V_CU(cudaMemcpy2DAsync(cols + row0, n * sizeof(fe), tails.data(), rows * sizeof(fe), rows * sizeof(fe), n_cols,
                             cudaMemcpyHostToDevice, pk->st));
    H2V_CU(cudaStreamSynchronize(pk->st));
    return H2V_OK;
}
int commit_dev(h2v_pk *pk, int basis, const fe *cols, size_t n_cols, std::vector<affine> &out) {
    out.resize(n_cols);
    if (!n_cols) return H2V_OK;
    H2V_TRY(pk->commits.ensure(n_cols * sizeof(affine)));
    H2V_TRY(h2v_commit_batch_dev(pk->srs, basis, cols, pk->n, n_cols, pk->n, pk->commits.p));
    H2V_CU(cudaSetDevice(pk->dev));
    H2V_CU(cudaMemcpy(out.data(), pk->commits.p, n_cols * sizeof(affine), cudaMemcpyDeviceToHost));
    return H2V_OK;
}
int write_points(PoseidonTranscript &T, const std::vector<affine> &pts) {
    for (const affine &p : pts)
        if (!T.write_point(p)) return failf(H2V_EINVAL, "create_proof: Cannot write points at infinity to the transcript");
    return H2V_OK;
}
struct PhaseClock {
    cudaEvent_t dummy;
    double t0;
    static double now() {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
    }
};

}  // namespace

extern "C" {

void h2v_pk_free(h2v_pk_t pk) {
    if (!pk) return;
    cudaSetDevice(pk->dev);
    DevBuf *all[] = {&pk->fixed_L, &pk->fixed_C, &pk->fixed_E, &pk->sigma_L, &pk->sigma_C, &pk->sigma_E, &pk->lrows_E, &pk->omega_pows,
                     &pk->adv_L, &pk->adv_C, &pk->adv_E, &pk->inst_L, &pk->inst_C, &pk->inst_E, &pk->pa_L, &pk->ps_L, &pk->pa_C, &pk->ps_C,
                     &pk->pa_E, &pk->ps_E, &pk->z_L, &pk->z_C, &pk->z_E, &pk->zl_L, &pk->zl_C, &pk->zl_E, &pk->num, &pk->den, &pk->tails,
                     &pk->ptrs, &pk->scal, &pk->pts, &pk->rnd_C, &pk->hq, &pk->hx_pieces, &pk->evals, &pk->pairs, &pk->sh_S, &pk->sh_A,
                     &pk->sh_B, &pk->sh_h, &pk->commits, &pk->scr_E, &pk->ext_cache};
    for (DevBuf *b : all) b->release();
    if (pk->dom) h2v_domain_free(pk->dom);
    if (pk->st) cudaStreamDestroy(pk->st);
    delete pk;
}

int h2v_pk_load(h2v_srs_t srs, const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma,
                const uint64_t vk_transcript_repr[4], h2v_pk_t *out) {
    if (!out) return failf(H2V_EINVAL, "pk_load: out is NULL");
    *out = nullptr;
    if (!srs || !cs || !vk_transcript_repr) return failf(H2V_EINVAL, "pk_load: NULL argument");
    if (cs->degree < 3 || cs->degree > 9) return failf(H2V_EINVAL, "pk_load: cs.degree() = %u unsupported", cs->degree);
    if (cs->k < 2 || cs->k > 24) return failf(H2V_EINVAL, "pk_load: k = %u unsupported", cs->k);
    const size_t n = (size_t)1 << cs->k;
    if ((size_t)cs->blinding_factors + 2 >= n) return failf(H2V_EINVAL, "pk_load: blinding_factors too large for k");
    if ((cs->n_fixed && !fixed) || (cs->n_perm && !sigma)) return failf(H2V_EINVAL, "pk_load: NULL column list");
    for (uint32_t j = 0; j < cs->n_gates; ++j)
        if (cs->gate_advice[j] >= cs->n_advice || cs->gate_selector[j] >= cs->n_fixed) return failf(H2V_EINVAL, "pk_load: gate %u out of range", j);
    for (uint32_t j = 0; j < cs->n_lookups; ++j)
        if (cs->lookup_input[j] >= cs->n_advice || cs->lookup_table[j] >= cs->n_fixed) return failf(H2V_EINVAL, "pk_load: lookup %u out of range", j);
    for (uint32_t j = 0; j < cs->n_perm; ++j) {
        const uint32_t lim = cs->perm_kind[j] == 0 ? cs->n_advice : cs->perm_kind[j] == 1 ? cs->n_fixed : cs->n_instance;
        if (cs->perm_kind[j] > 2 || cs->perm_index[j] >= lim) return failf(H2V_EINVAL, "pk_load: permutation column %u out of range", j);
    }
    for (uint32_t j = 0; j < cs->n_advice_queries; ++j)
        if (cs->advice_query_col[j] >= cs->n_advice) return failf(H2V_EINVAL, "pk_load: advice query %u out of range", j);
    for (uint32_t j = 0; j < cs->n_fixed_queries; ++j)
        if (cs->fixed_query_col[j] >= cs->n_fixed) return failf(H2V_EINVAL, "pk_load: fixed query %u out of range", j);
    uint32_t srs_c = 0;
    H2V_TRY(h2v_srs_info(srs, &srs_c, nullptr));

    if (cudaSetDevice(current_device()) != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ECUDA, "pk_load: no CUDA device (libh2v has no CPU fallback)");
    }
    h2v_pk *pk = new h2v_pk();
    pk->dev = current_device();
    pk->srs = srs;
    pk->k = cs->k; pk->degree = cs->degree; pk->bf = cs->blinding_factors;
    pk->n_advice = cs->n_advice; pk->n_fixed = cs->n_fixed; pk->n_instance = cs->n_instance;
    pk->gate_advice.assign(cs->gate_advice, cs->gate_advice + cs->n_gates);
    pk->gate_selector.assign(cs->gate_selector, cs->gate_selector + cs->n_gates);
    pk->lookup_input.assign(cs->lookup_input, cs->lookup_input + cs->n_lookups);
    pk->lookup_table.assign(cs->lookup_table, cs->lookup_table + cs->n_lookups);
    pk->perm_kind.assign(cs->perm_kind, cs->perm_kind + cs->n_perm);
    pk->perm_index.assign(cs->perm_index, cs->perm_index + cs->n_perm);
    pk->aq_col.assign(cs->advice_query_col, cs->advice_query_col + cs->n_advice_queries);
    pk->aq_rot.assign(cs->advice_query_rot, cs->advice_query_rot + cs->n_advice_queries);
    pk->fq_col.assign(cs->fixed_query_col, cs->fixed_query_col + cs->n_fixed_queries);
    pk->fq_rot.assign(cs->fixed_query_rot, cs->fixed_query_rot + cs->n_fixed_queries);
    pk->n = n;
    pk->u = (uint32_t)(n - (cs->blinding_factors + 1));
    pk->chunk = cs->degree - 2;
    pk->n_sets = cs->n_perm ? (cs->n_perm + pk->chunk - 1) / pk->chunk : 0;
    pk->vk_repr = frh::load(vk_transcript_repr);
    int rc = h2v_domain_new(cs->degree, cs->k, &pk->dom);
    if (rc) { h2v_pk_free(pk); return rc; }
    pk->ne = (size_t)1 << h2v_domain_extended_k(pk->dom);
    uint64_t tmp[4];
    h2v_domain_constant(pk->dom, 0, tmp); pk->omega = frh::load(tmp);
    h2v_domain_constant(pk->dom, 1, tmp); pk->omega_inv = frh::load(tmp);
    pk->delta = frh::pow_u64(frh::from_u64(7), (uint64_t)1 << 28);      // Fr::DELTA = MULTIPLICATIVE_GENERATOR^(2^S)
    cudaSetDevice(pk->dev);      // h2v_domain_new built one replica per device and left this thread on the last one
    cudaError_t e = cudaStreamCreateWithFlags(&pk->st, cudaStreamNonBlocking);
    if (e != cudaSuccess) { h2v_pk_free(pk); return failf(H2V_ECUDA, "pk_load: %s", cudaGetErrorString(e)); }

    {
        // everything resident (the default): Lagrange, coefficient and extended forms of every column of the key and of the
        // proof.  When that exceeds about half of the device's memory (SIFT-shaped k = 20: 204 GB), stream the extended forms.
        size_t free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        const double cols = (double)cs->n_fixed + cs->n_perm + cs->n_advice + cs->n_instance + 3.0 * cs->n_lookups + pk->n_sets;
        const double resident = cols * (2.0 * n + (double)pk->ne) * sizeof(fe);
        const char *e = getenv("H2V_STREAM_EXT");
        pk->stream_ext = e ? atoi(e) != 0 : resident > 0.55 * (double)total_b;
        const char *ec = getenv("H2V_STREAM_COLS");
        const size_t want = ec ? (size_t)atoi(ec) : ((size_t)12 << 30) / (pk->ne * sizeof(fe));
        pk->scr_cols = std::min<size_t>(std::max<size_t>(want, 2 * (size_t)pk->chunk + 2), 512);
    }
    auto body = [&]() -> int {
        const size_t ne = pk->ne;
        // fixed columns and sigma polynomials: Lagrange (as given) -> coefficients -> extended coset, all resident
        struct Grp { const uint64_t *const *src; size_t cnt; DevBuf *L, *C, *E; } grp[2] = {
            {fixed, cs->n_fixed, &pk->fixed_L, &pk->fixed_C, &pk->fixed_E}, {sigma, cs->n_perm, &pk->sigma_L, &pk->sigma_C, &pk->sigma_E}};
        for (auto &g : grp) {
            if (!g.cnt) continue;
            H2V_TRY(g.L->ensure(g.cnt * n * sizeof(fe)));
            H2V_TRY(g.C->ensure(g.cnt * n * sizeof(fe)));
            if (!pk->stream_ext) H2V_TRY(g.E->ensure(g.cnt * ne * sizeof(fe)));
            for (size_t c = 0; c < g.cnt; ++c) {
                if (!g.src[c]) return failf(H2V_EINVAL, "pk_load: column %zu is NULL", c);
                H2V_CU(cudaMemcpyAsync(g.L->as<fe>() + c * n, g.src[c], n * sizeof(fe), cudaMemcpyHostToDevice, pk->st));
            }
            H2V_TRY(sync(pk));
            H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_LAGRANGE_TO_COEFF, g.L->p, n, g.C->p, n, g.cnt));
            if (!pk->stream_ext) H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_COEFF_TO_EXTENDED, g.C->p, n, g.E->p, ne, g.cnt));
        }
        // l_0, l_last, l_active_row = 1 - (l_last + l_blind) on the extended coset (keygen.rs)
        {
            std::vector<Fr64> rows(3 * n, frh::zero());
            rows[0] = frh::ONE;                                    // l_0
            rows[n + pk->u] = frh::ONE;                            // l_last: row n - blinding_factors - 1
            for (size_t i = 0; i < pk->u; ++i) rows[2 * n + i] = frh::ONE;      // active rows
            DevBuf L, Cf;
            H2V_TRY(L.ensure(3 * n * sizeof(fe)));
            int rc2 = Cf.ensure(3 * n * sizeof(fe));
            if (!rc2) rc2 = pk->lrows_E.ensure(3 * ne * sizeof(fe));
            if (!rc2 && cudaMemcpy(L.p, rows.data(), 3 * n * sizeof(fe), cudaMemcpyHostToDevice) != cudaSuccess)
                rc2 = failf(H2V_ECUDA, "pk_load: upload failed");
            if (!rc2) rc2 = h2v_domain_transform_dev(pk->dom, H2V_OP_LAGRANGE_TO_COEFF, L.p, n, Cf.p, n, 3);
            if (!rc2) rc2 = h2v_domain_transform_dev(pk->dom, H2V_OP_COEFF_TO_EXTENDED, Cf.p, n, pk->lrows_E.p, ne, 3);
            L.release();
            Cf.release();
            if (rc2) return rc2;
        }
        // w^i for the permutation numerators
        {
            std::vector<Fr64> pw(n);
            Fr64 cur = frh::ONE;
            for (size_t i = 0; i < n; ++i) {
                pw[i] = cur;
                cur = frh::mul(cur, pk->omega);
            }
            H2V_TRY(pk->omega_pows.ensure(n * sizeof(fe)));
            H2V_CU(cudaMemcpy(pk->omega_pows.p, pw.data(), n * sizeof(fe), cudaMemcpyHostToDevice));
        }
        return H2V_OK;
    };
    rc = body();
    if (rc) { h2v_pk_free(pk); return rc; }
    *out = pk;
    return H2V_OK;
}

int h2v_pk_last_phase_ms(h2v_pk_t pk, double out[8]) {
    if (!pk || !out) return failf(H2V_EINVAL, "pk_last_phase_ms: NULL argument");
    memcpy(out, pk->last_ms, sizeof pk->last_ms);
    return H2V_OK;
}

}  // extern "C"

// ================================================================== create_proof
namespace {

struct Query {
    const fe *poly;     // device-resident coefficients (n): the commitment's identity, as upstream's PolynomialPointer
    uint32_t pt;        // index into the distinct evaluation points
    Fr64 eval;
};

int create_proof_locked(h2v_pk *pk, const uint64_t *const *advice, const uint64_t *const *instances, const uint32_t *instance_len,
                        const uint8_t rng_seed[32], std::vector<uint8_t> &proof) {
    const size_t n = pk->n, ne = pk->ne;
    const uint32_t A = pk->n_advice, F = pk->n_fixed, I = pk->n_instance, L = (uint32_t)pk->lookup_input.size(),
                   G = (uint32_t)pk->gate_advice.size(), NP = (uint32_t)pk->perm_kind.size(), NS = pk->n_sets, bf = pk->bf, u = pk->u;
    const unsigned gn = (unsigned)((n + 255) / 256);
    cudaStream_t st = pk->st;
    double t_phase = PhaseClock::now();
    int phase = 0;
    auto lap = [&]() {
        double t = PhaseClock::now();
        if (phase < 8) pk->last_ms[phase++] = t - t_phase;
        t_phase = t;
    };
    for (double &v : pk->last_ms) v = 0;

    PoseidonTranscript T;
    ChaCha20Rng rng(rng_seed);
    // ---- 1. vk, instances                                                   (prover.rs: hash_into, common_scalar)
    T.common_scalar(pk->vk_repr);
    H2V_TRY(pk->inst_L.ensure(std::max<size_t>(1, I) * n * sizeof(fe)));
    H2V_TRY(pk->inst_C.ensure(std::max<size_t>(1, I) * n * sizeof(fe)));
    H2V_TRY(pk->inst_E.ensure(std::max<size_t>(1, I) * ne * sizeof(fe)));
    if (I) {
        std::vector<Fr64> inst(I * n, frh::zero());
        for (uint32_t c = 0; c < I; ++c) {
            if (instance_len[c] > u) return failf(H2V_EINVAL, "create_proof: InstanceTooLarge (%u values, %u usable rows)", instance_len[c], u);
            for (uint32_t i = 0; i < instance_len[c]; ++i) {
                inst[c * n + i] = frh::load(instances[c] + 4 * i);
                T.common_scalar(inst[c * n + i]);
            }
        }
        H2V_TRY(upload(pk, pk->inst_L, 0, inst.data(), I * n * sizeof(fe)));
        H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_LAGRANGE_TO_COEFF, pk->inst_L.p, n, pk->inst_C.p, n, I));
    }
    // ---- 2-4. advice columns: upload, blind the last blinding_factors + 1 rows, commit
    H2V_TRY(pk->adv_L.ensure((size_t)A * n * sizeof(fe)));
    H2V_TRY(pk->adv_C.ensure((size_t)A * n * sizeof(fe)));
    for (uint32_t c = 0; c < A; ++c)
        if (!advice[c]) return failf(H2V_EINVAL, "create_proof: advice[%u] is NULL", c);
    // h2v_commit_batch_resident: each device uploads its block of the columns in sub-batches (the next one crosses while the
    // previous one is committed), writes the tails, commits the block and leaves it in adv_L
    std::vector<Fr64> tails((size_t)A * (bf + 1));
    for (auto &t : tails) t = rng.fr_random();                       // column by column, rows u .. n-1
    for (uint32_t c = 0; c < A; ++c) (void)rng.fr_random();          // one Blind per column (unused by KZG, but drawn)
    std::vector<affine> pts(A);
    H2V_TRY(h2v_commit_batch_resident(pk->srs, H2V_BASIS_LAGRANGE, advice, A, n, (const uint64_t *)tails.data(), u, bf + 1, pk->adv_L.p, n,
                                      (uint64_t *)pts.data()));
    H2V_CU(cudaSetDevice(pk->dev));
    H2V_TRY(write_points(T, pts));
    T.absorb_async();      // the advice commitments are hashed on a worker thread while the lookup permutations run
    lap();   // phase 0: upload + advice commitments
    // column pointer helpers
    auto col_L = [&](uint8_t kind, uint32_t idx) -> const fe * {
        return kind == 0 ? pk->adv_L.as<fe>() + (size_t)idx * n : kind == 1 ? pk->fixed_L.as<fe>() + (size_t)idx * n : pk->inst_L.as<fe>() + (size_t)idx * n;
    };
    auto col_E = [&](uint8_t kind, uint32_t idx) -> const fe * {
        return kind == 0 ? pk->adv_E.as<fe>() + (size_t)idx * ne : kind == 1 ? pk->fixed_E.as<fe>() + (size_t)idx * ne : pk->inst_E.as<fe>() + (size_t)idx * ne;
    };
    // ---- 5. theta; lookups: permuted input / table columns                   (lookup/prover.rs commit_permuted)
    // theta is squeezed at its place in the transcript (below, before A' / S' are written); single-expression lookups
    // have nothing to compress, so the permutations do not wait for it
    H2V_TRY(pk->pa_L.ensure(std::max<size_t>(1, L) * n * sizeof(fe)));
    H2V_TRY(pk->ps_L.ensure(std::max<size_t>(1, L) * n * sizeof(fe)));
    if (L) {
        std::vector<Fr64> ta((size_t)L * (bf + 1)), ts((size_t)L * (bf + 1));
        {
            std::vector<const void *> li(L), lt(L);
            for (uint32_t l = 0; l < L; ++l) {
                li[l] = col_L(0, pk->lookup_input[l]);
                lt[l] = col_L(1, pk->lookup_table[l]);
            }
            H2V_TRY(h2v_permute_expression_pair_batch_dev(li.data(), lt.data(), L, u, pk->pa_L.as<fe>(), n, pk->ps_L.as<fe>(), n));
            H2V_CU(cudaSetDevice(pk->dev));
        }
        for (uint32_t l = 0; l < L; ++l) {
            for (uint32_t i = 0; i <= bf; ++i) ta[(size_t)l * (bf + 1) + i] = rng.fr_random();
            for (uint32_t i = 0; i <= bf; ++i) ts[(size_t)l * (bf + 1) + i] = rng.fr_random();
            (void)rng.fr_random();     // permuted input blind
            (void)rng.fr_random();     // permuted table blind
        }
        H2V_TRY(write_rows(pk, pk->pa_L.as<fe>(), n, u, bf + 1, L, ta));
        H2V_TRY(write_rows(pk, pk->ps_L.as<fe>(), n, u, bf + 1, L, ts));
        std::vector<affine> ca, cs_;
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->pa_L.as<fe>(), L, ca));
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->ps_L.as<fe>(), L, cs_));
        (void)T.squeeze_challenge();      // theta
        for (uint32_t l = 0; l < L; ++l) {
            if (!T.write_point(ca[l]) || !T.write_point(cs_[l]))
                return failf(H2V_EINVAL, "create_proof: Cannot write points at infinity to the transcript");
        }
    }
    else (void)T.squeeze_challenge();     // theta
    lap();   // phase 1: lookup permutations
    // ---- 6. beta, gamma; permutation grand products                          (permutation/prover.rs commit)
    const Fr64 beta = T.squeeze_challenge(), gamma = T.squeeze_challenge();
    H2V_TRY(pk->z_L.ensure(std::max<size_t>(1, NS) * n * sizeof(fe)));
    H2V_TRY(pk->num.ensure(std::max<size_t>(1, std::max(NS, L)) * n * sizeof(fe)));
    H2V_TRY(pk->den.ensure(std::max<size_t>(1, std::max(NS, L)) * n * sizeof(fe)));
    H2V_TRY(pk->ptrs.ensure((size_t)(4 * (NP + G + L) + 4096) * sizeof(void *)));
    H2V_TRY(pk->scal.ensure((size_t)(NS + A + F + NP + 3 * NS + 5 * L + 64) * sizeof(fe) + 4096));
    if (NS) {
        std::vector<const fe *> hp(2 * NP);
        for (uint32_t c = 0; c < NP; ++c) {
            hp[c] = col_L(pk->perm_kind[c], pk->perm_index[c]);
            hp[NP + c] = pk->sigma_L.as<fe>() + (size_t)c * n;
        }
        H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
        std::vector<Fr64> dstart(NS);
        const Fr64 dchunk = frh::pow_u64(pk->delta, pk->chunk);
        Fr64 cur = frh::ONE;
        for (uint32_t s = 0; s < NS; ++s) {
            dstart[s] = cur;
            cur = frh::mul(cur, dchunk);
        }
        H2V_TRY(upload(pk, pk->scal, 0, dstart.data(), NS * sizeof(fe)));
        PermArgs pa;
        pa.cols = (const fe *const *)pk->ptrs.p;
        pa.sigma = pa.cols + NP;
        pa.omega_pows = pk->omega_pows.as<fe>();
        pa.delta_start = pk->scal.as<fe>();
        pa.beta = frh::to_fe(beta); pa.gamma = frh::to_fe(gamma); pa.delta = frh::to_fe(pk->delta);
        pa.n_cols = NP; pa.chunk = pk->chunk; pa.n = (uint32_t)n;
        perm_numden_kernel<<<dim3(gn, NS), 256, 0, st>>>(pa, pk->num.as<fe>(), pk->den.as<fe>());
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        // z_s with z_s[0] = 1; then chain: z_s *= z_{s-1}[u] (upstream carries `last_z` from set to set)
        H2V_TRY(h2v_grand_product_dev(pk->num.p, pk->den.p, n, NS, pk->z_L.p));
        std::vector<Fr64> last(NS), scale(NS);
        H2V_CU(cudaMemcpy2D(last.data(), sizeof(fe), pk->z_L.as<fe>() + u, n * sizeof(fe), sizeof(fe), NS, cudaMemcpyDeviceToHost));
        cur = frh::ONE;
        for (uint32_t s = 0; s < NS; ++s) {
            scale[s] = cur;
            cur = frh::mul(cur, last[s]);
        }
        H2V_TRY(upload(pk, pk->scal, 0, scale.data(), NS * sizeof(fe)));
        scale_cols_kernel<<<dim3(gn, NS), 256, 0, st>>>(pk->z_L.as<fe>(), (uint32_t)n, pk->scal.as<fe>());
        H2V_LAUNCHED();
        std::vector<Fr64> tails((size_t)NS * bf);
        for (uint32_t s = 0; s < NS; ++s) {
            for (uint32_t i = 0; i < bf; ++i) tails[(size_t)s * bf + i] = rng.fr_random();     // rows n - bf .. n - 1
            (void)rng.fr_random();                                                             // product blind
        }
        H2V_TRY(write_rows(pk, pk->z_L.as<fe>(), n, n - bf, bf, NS, tails));
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->z_L.as<fe>(), NS, pts));
        H2V_TRY(write_points(T, pts));
        T.absorb_async();      // hashed while the lookup products are built and committed
    }
    // ---- 7. lookup grand products                                             (lookup/prover.rs commit_product)
    H2V_TRY(pk->zl_L.ensure(std::max<size_t>(1, L) * n * sizeof(fe)));
    if (L) {
        std::vector<const fe *> hp(2 * L);
        for (uint32_t l = 0; l < L; ++l) {
            hp[l] = col_L(0, pk->lookup_input[l]);
            hp[L + l] = col_L(1, pk->lookup_table[l]);
        }
        H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
        lookup_numden_kernel<<<dim3(gn, L), 256, 0, st>>>((const fe *const *)pk->ptrs.p, (const fe *const *)pk->ptrs.p + L, pk->pa_L.as<fe>(),
                                                        pk->ps_L.as<fe>(), frh::to_fe(beta), frh::to_fe(gamma), (uint32_t)n, pk->num.as<fe>(), pk->den.as<fe>());
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        H2V_TRY(h2v_grand_product_dev(pk->num.p, pk->den.p, n, L, pk->zl_L.p));
        std::vector<Fr64> tails((size_t)L * bf);
        for (uint32_t l = 0; l < L; ++l) {
            for (uint32_t i = 0; i < bf; ++i) tails[(size_t)l * bf + i] = rng.fr_random();
            (void)rng.fr_random();
        }
        H2V_TRY(write_rows(pk, pk->zl_L.as<fe>(), n, n - bf, bf, L, tails));
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->zl_L.as<fe>(), L, pts));
        H2V_TRY(write_points(T, pts));
        T.absorb_async();
    }
    lap();   // phase 2: grand products
    // ---- 8. vanishing argument: random polynomial                             (vanishing/prover.rs commit)
    H2V_TRY(pk->rnd_C.ensure(n * sizeof(fe)));
    {
        // n consecutive Fr::random draws = n consecutive key-stream blocks: produced on the device
        ChaChaKey key;
        memcpy(key.k, rng.key, 32);
        chacha_fr_kernel<<<gn, 256, 0, st>>>(key, rng.next_block(), (uint32_t)n, pk->rnd_C.as<fe>());
        H2V_LAUNCHED();
        rng.skip_fr(n);
        (void)rng.fr_random();      // random_blind
        H2V_TRY(sync(pk));
        H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, pk->rnd_C.as<fe>(), 1, pts));
        H2V_TRY(write_points(T, pts));
        T.absorb_async();
    }
    // ---- 9-11. coefficient and extended forms (no challenge involved: they run while the commitments above are hashed);
    //            then y, evaluate_h, quotient pieces
    const int L2C = H2V_OP_LAGRANGE_TO_COEFF, C2E = H2V_OP_COEFF_TO_EXTENDED;
    const bool stream = pk->stream_ext;
    // (the per-proof buffers are kept between proofs, also in streamed mode: with peer access enabled, freeing and
    // re-allocating gigabytes every proof costs more than the transforms themselves -- measured on two devices)
    if (!stream) H2V_TRY(pk->adv_E.ensure((size_t)A * ne * sizeof(fe)));
    H2V_TRY(h2v_domain_transform_dev(pk->dom, L2C, pk->adv_L.p, n, pk->adv_C.p, n, A));
    if (!stream) H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, pk->adv_C.p, n, pk->adv_E.p, ne, A));
    if (I) H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, pk->inst_C.p, n, pk->inst_E.p, ne, I));
    struct Tr { DevBuf *Lb, *Cb, *Eb; size_t cnt; } trs[4] = {{&pk->pa_L, &pk->pa_C, &pk->pa_E, L}, {&pk->ps_L, &pk->ps_C, &pk->ps_E, L},
                                                            {&pk->z_L, &pk->z_C, &pk->z_E, NS}, {&pk->zl_L, &pk->zl_C, &pk->zl_E, L}};
    for (auto &t : trs) {
        H2V_TRY(t.Cb->ensure(std::max<size_t>(1, t.cnt) * n * sizeof(fe)));
        H2V_TRY(t.Eb->ensure(std::max<size_t>(1, t.cnt) * ne * sizeof(fe)));
        if (!t.cnt) continue;
        H2V_TRY(h2v_domain_transform_dev(pk->dom, L2C, t.Lb->p, n, t.Cb->p, n, t.cnt));
        H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, t.Cb->p, n, t.Eb->p, ne, t.cnt));
    }
    const Fr64 y = T.squeeze_challenge();
    lap();   // phase 3: random poly + transforms
    H2V_TRY(pk->hq.ensure(2 * ne * sizeof(fe)));
    fe *h_ext = pk->hq.as<fe>(), *h_out = pk->hq.as<fe>() + ne;
    H2V_CU(cudaMemsetAsync(h_ext, 0, ne * sizeof(fe), st));
    H2V_TRY(sync(pk));
    const fe *l0 = pk->lrows_E.as<fe>(), *ll = l0 + ne, *la = l0 + 2 * ne;
    if (!stream) {
        std::vector<const fe *> hp(2 * G + 2 * NP);
        for (uint32_t j = 0; j < G; ++j) {
            hp[j] = col_E(1, pk->gate_selector[j]);
            hp[G + j] = col_E(0, pk->gate_advice[j]);
        }
        for (uint32_t c = 0; c < NP; ++c) {
            hp[2 * G + c] = col_E(pk->perm_kind[c], pk->perm_index[c]);
            hp[2 * G + NP + c] = pk->sigma_E.as<fe>() + (size_t)c * ne;
        }
        if (!hp.empty()) H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
        const void *const *tab = (const void *const *)pk->ptrs.p;
        H2V_TRY(h2v_quotient_gates_ptrs_dev(pk->dom, h_ext, u64(y), G, tab, tab + G));
        if (NP)
            H2V_TRY(h2v_quotient_permutation_ptrs_dev(pk->dom, h_ext, u64(y), u64(beta), u64(gamma), NP, pk->chunk, tab + 2 * G,
                                                      tab + 2 * G + NP, pk->z_E.p, ne, l0, ll, la, bf));
        for (uint32_t l = 0; l < L; ++l)
            H2V_TRY(h2v_quotient_lookup_dev(pk->dom, h_ext, u64(y), u64(beta), u64(gamma), col_E(0, pk->lookup_input[l]),
                                            col_E(1, pk->lookup_table[l]), pk->pa_E.as<fe>() + (size_t)l * ne, pk->ps_E.as<fe>() + (size_t)l * ne,
                                            pk->zl_E.as<fe>() + (size_t)l * ne, l0, ll, la));
    } else {
        // the same folds, in upstream's order, over slices of columns whose extended forms are rebuilt into `scr_E` from
        // the resident coefficient forms (every term reads columns of its own gate / set / lookup only)
        const size_t SC = pk->scr_cols;
        H2V_TRY(pk->scr_E.ensure(SC * ne * sizeof(fe)));
        fe *scr = pk->scr_E.as<fe>();
        auto col_C = [&](uint8_t kind, uint32_t idx) -> const fe * {
            return kind == 0 ? pk->adv_C.as<fe>() + (size_t)idx * n : kind == 1 ? pk->fixed_C.as<fe>() + (size_t)idx * n : pk->inst_C.as<fe>() + (size_t)idx * n;
        };
        // coeff_to_extended of a list of coefficient columns into consecutive scratch slots; neighbours share one launch
        const bool timing = getenv("H2V_PROVE_TIMING") != nullptr;
        double t_ext = 0, t_fold = 0, t_mark = PhaseClock::now();
        auto mark = [&](double &acc) {
            if (!timing) return;
            cudaDeviceSynchronize();
            const double t = PhaseClock::now();
            acc += t - t_mark;
            t_mark = t;
        };
        auto extend = [&](const std::vector<const fe *> &src, fe *dst) -> int {
            for (size_t i = 0; i < src.size();) {
                size_t j = i + 1;
                while (j < src.size() && src[j] == src[j - 1] + n) ++j;
                H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, src[i], n, dst + i * ne, ne, j - i));
                i = j;
            }
            return H2V_OK;
        };
        const void *const *tab = (const void *const *)pk->ptrs.p;
        std::vector<const fe *> src, hp;
        // Gate j reads one advice column, and (in halo2-base's constraint system) every gate column is also a permutation
        // column: when the gates meet their columns in gate order along the permutation, one pass over the permutation
        // slices serves both folds -- the gates into h, the permutation into a second accumulator hp (the memory of the
        // quotient's output, free until the division), joined as h <- h y^(permutation terms) + hp.  Each advice column is
        // then extended once instead of twice.  Any other constraint system takes the two separate loops below.
        std::vector<int32_t> gate_of_adv(A, -1);
        for (uint32_t j = 0; j < G; ++j) gate_of_adv[pk->gate_advice[j]] = gate_of_adv[pk->gate_advice[j]] == -1 ? (int32_t)j : -2;
        bool fused = NP > 0 && G > 0;
        {
            uint32_t next_gate = 0;
            for (uint32_t c = 0; c < NP && fused; ++c)
                if (pk->perm_kind[c] == 0 && gate_of_adv[pk->perm_index[c]] != -1) fused = gate_of_adv[pk->perm_index[c]] == (int32_t)next_gate++;
            fused = fused && next_gate == G;
        }
        if (fused) {
            fe *hp_acc = h_out;
            H2V_CU(cudaMemsetAsync(hp_acc, 0, ne * sizeof(fe), st));
            H2V_TRY(sync(pk));
            if (!pk->cache_tried) {
                pk->cache_tried = true;
                size_t free_b = 0, total_b = 0;
                cudaMemGetInfo(&free_b, &total_b);
                const char *e = getenv("H2V_EXT_CACHE_COLS");
                const size_t margin = (size_t)8 << 30;
                size_t want = e ? (size_t)atoi(e) : (free_b > margin ? (free_b - margin) / (ne * sizeof(fe)) : 0);
                want = std::min<size_t>(want, NP);
                if (want >= (e ? 1u : 8u) && pk->ext_cache.ensure(want * ne * sizeof(fe)) == H2V_OK) {
                    H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, pk->sigma_C.p, n, pk->ext_cache.p, ne, want));
                    pk->cached_sigma = want;
                }
            }
            const size_t BS = std::max<size_t>(1, SC / (3 * (size_t)pk->chunk));
            std::vector<const fe *> pc, sg, gq, ga;
            for (size_t s0 = 0; s0 < NS; s0 += BS) {
                const size_t s1 = std::min<size_t>(NS, s0 + BS), c0 = s0 * pk->chunk, c1 = std::min<size_t>(NP, s1 * pk->chunk), cnt = c1 - c0;
                src.clear(); pc.clear(); sg.clear(); gq.clear(); ga.clear();
                size_t slot = 0;
                for (size_t c = c0; c < c1; ++c) {
                    src.push_back(col_C(pk->perm_kind[c], pk->perm_index[c]));
                    pc.push_back(scr + slot++ * ne);
                }
                for (size_t c = c0; c < c1; ++c) {
                    if (c < pk->cached_sigma) {
                        sg.push_back(pk->ext_cache.as<fe>() + c * ne);
                    } else {
                        src.push_back(pk->sigma_C.as<fe>() + c * n);
                        sg.push_back(scr + slot++ * ne);
                    }
                }
                // this slice's gates: selector extended behind the slice, advice already in it
                for (size_t c = c0; c < c1; ++c) {
                    if (pk->perm_kind[c] != 0 || gate_of_adv[pk->perm_index[c]] < 0) continue;
                    src.push_back(col_C(1, pk->gate_selector[gate_of_adv[pk->perm_index[c]]]));
                    gq.push_back(scr + slot++ * ne);
                    ga.push_back(pc[c - c0]);
                }
                H2V_TRY(extend(src, scr));
                mark(t_ext);
                hp.clear();
                hp.insert(hp.end(), pc.begin(), pc.end());
                hp.insert(hp.end(), sg.begin(), sg.end());
                hp.insert(hp.end(), gq.begin(), gq.end());
                hp.insert(hp.end(), ga.begin(), ga.end());
                H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
                H2V_TRY(h2v_quotient_permutation_range_ptrs_dev(pk->dom, hp_acc, u64(y), u64(beta), u64(gamma), NP, pk->chunk, s0, s1, s0 == 0,
                                                                tab, tab + cnt, pk->z_E.p, ne, l0, ll, la, bf));
                if (!gq.empty()) H2V_TRY(h2v_quotient_gates_ptrs_dev(pk->dom, h_ext, u64(y), gq.size(), tab + 2 * cnt, tab + 2 * cnt + gq.size()));
                mark(t_fold);
            }
            // h <- h y^T + hp, T = the permutation argument's terms: 2 + (NS - 1) + NS
            const fe *two[2] = {h_ext, hp_acc};
            const Fr64 cf[2] = {frh::pow_u64(y, 2ull * NS + 1), frh::ONE};
            H2V_TRY(upload(pk, pk->ptrs, 0, two, sizeof two));
            H2V_TRY(upload(pk, pk->scal, 0, cf, sizeof cf));
            lincomb_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>((const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), 2, (uint32_t)ne, h_ext);
            H2V_LAUNCHED();
            H2V_TRY(sync(pk));
            mark(t_fold);
        } else {
        const size_t BG = SC / 2;
        for (size_t g0 = 0; g0 < G; g0 += BG) {
            const size_t b = std::min<size_t>(BG, G - g0);
            src.clear();
            hp.assign(2 * b, nullptr);
            for (size_t j = 0; j < b; ++j) src.push_back(col_C(1, pk->gate_selector[g0 + j]));
            for (size_t j = 0; j < b; ++j) src.push_back(col_C(0, pk->gate_advice[g0 + j]));
            H2V_TRY(extend(src, scr));
            mark(t_ext);
            for (size_t j = 0; j < 2 * b; ++j) hp[j] = scr + j * ne;
            H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
            H2V_TRY(h2v_quotient_gates_ptrs_dev(pk->dom, h_ext, u64(y), b, tab, tab + b));
            mark(t_fold);
        }
        const size_t BS = std::max<size_t>(1, SC / (2 * (size_t)pk->chunk));
        for (size_t s0 = 0; s0 < NS; s0 += BS) {
            const size_t s1 = std::min<size_t>(NS, s0 + BS), c0 = s0 * pk->chunk, c1 = std::min<size_t>(NP, s1 * pk->chunk), cnt = c1 - c0;
            src.clear();
            hp.assign(2 * cnt, nullptr);
            for (size_t c = c0; c < c1; ++c) src.push_back(col_C(pk->perm_kind[c], pk->perm_index[c]));
            for (size_t c = c0; c < c1; ++c) src.push_back(pk->sigma_C.as<fe>() + c * n);
            H2V_TRY(extend(src, scr));
            mark(t_ext);
            for (size_t j = 0; j < 2 * cnt; ++j) hp[j] = scr + j * ne;
            H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), hp.size() * sizeof(void *)));
            H2V_TRY(h2v_quotient_permutation_range_ptrs_dev(pk->dom, h_ext, u64(y), u64(beta), u64(gamma), NP, pk->chunk, s0, s1, s0 == 0,
                                                            tab, tab + cnt, pk->z_E.p, ne, l0, ll, la, bf));
            mark(t_fold);
        }
        }
        // lookups: the table's extended form in slot 0 (one table for all of halo2-base's range lookups), the inputs of up
        // to SC - 1 lookups extended together (a single 2^22-point column transforms four times slower per column than a batch)
        uint32_t table_in_slot = UINT32_MAX;
        for (uint32_t l0_ = 0; l0_ < L;) {
            if (pk->lookup_table[l0_] != table_in_slot) {
                H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, col_C(1, pk->lookup_table[l0_]), n, scr, ne, 1));
                table_in_slot = pk->lookup_table[l0_];
            }
            uint32_t l1_ = l0_;
            src.clear();
            while (l1_ < L && pk->lookup_table[l1_] == table_in_slot && src.size() + 1 < SC) src.push_back(col_C(0, pk->lookup_input[l1_++]));
            H2V_TRY(extend(src, scr + ne));
            mark(t_ext);
            for (uint32_t l = l0_; l < l1_; ++l)
                H2V_TRY(h2v_quotient_lookup_dev(pk->dom, h_ext, u64(y), u64(beta), u64(gamma), scr + (size_t)(1 + l - l0_) * ne, scr,
                                                pk->pa_E.as<fe>() + (size_t)l * ne, pk->ps_E.as<fe>() + (size_t)l * ne, pk->zl_E.as<fe>() + (size_t)l * ne, l0, ll, la));
            mark(t_fold);
            l0_ = l1_;
        }
        if (timing) fprintf(stderr, "evaluate_h (streamed): coeff_to_extended of the slices %.1f ms, folds %.1f ms\n", t_ext, t_fold);
    }
    H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_DIVIDE_BY_VANISHING, h_ext, ne, h_out, ne, 1));
    const uint32_t NH = pk->degree - 1;          // quotient pieces of n coefficients each
    for (uint32_t i = 0; i < NH; ++i) (void)rng.fr_random();     // h_blinds
    H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, h_out, NH, pts));
    H2V_TRY(write_points(T, pts));
    lap();   // phase 4: evaluate_h + quotient commitments
    // ---- 12. x; evaluations
    const Fr64 x = T.squeeze_challenge();
    Fr64 xn = x;
    for (uint32_t i = 0; i < pk->k; ++i) xn = frh::sqr(xn);
    // distinct evaluation points x * w^rot
    std::vector<int32_t> rots;
    std::vector<Fr64> points;
    auto point_of = [&](int32_t rot) -> uint32_t {
        for (size_t i = 0; i < rots.size(); ++i)
            if (rots[i] == rot) return (uint32_t)i;
        rots.push_back(rot);
        points.push_back(frh::rotate(x, pk->omega, pk->omega_inv, rot));
        return (uint32_t)(rots.size() - 1);
    };
    const uint32_t p_cur = point_of(0), p_next = point_of(1), p_prev = point_of(-1), p_last = point_of(-(int32_t)(bf + 1));
    // h(X) = sum_i xn^i h_i(X)
    H2V_TRY(pk->sh_h.ensure(2 * n * sizeof(fe)));
    fe *h_poly = pk->sh_h.as<fe>(), *hx_dev = pk->sh_h.as<fe>() + n;
    {
        std::vector<const fe *> hp(NH);
        std::vector<Fr64> cf(NH);
        Fr64 cur = frh::ONE;
        for (uint32_t i = 0; i < NH; ++i) {
            hp[i] = h_out + (size_t)i * n;
            cf[i] = cur;
            cur = frh::mul(cur, xn);
        }
        H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), NH * sizeof(void *)));
        H2V_TRY(upload(pk, pk->scal, 0, cf.data(), NH * sizeof(fe)));
        lincomb_kernel<<<gn, 256, 0, st>>>((const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), NH, (uint32_t)n, h_poly);
        H2V_LAUNCHED();
    }
    // every (polynomial, point) pair that is evaluated, in transcript order first, then the two the transcript skips
    std::vector<EvalPair> pairs;
    auto push = [&](const fe *poly, uint32_t pt) { pairs.push_back(EvalPair{poly, pt}); return (uint32_t)(pairs.size() - 1); };
    for (size_t q = 0; q < pk->aq_col.size(); ++q) push(pk->adv_C.as<fe>() + (size_t)pk->aq_col[q] * n, point_of(pk->aq_rot[q]));
    for (size_t q = 0; q < pk->fq_col.size(); ++q) push(pk->fixed_C.as<fe>() + (size_t)pk->fq_col[q] * n, point_of(pk->fq_rot[q]));
    const uint32_t e_random = push(pk->rnd_C.as<fe>(), p_cur);
    for (uint32_t c = 0; c < NP; ++c) push(pk->sigma_C.as<fe>() + (size_t)c * n, p_cur);
    const uint32_t e_perm = (uint32_t)pairs.size();
    for (uint32_t s = 0; s < NS; ++s) {
        push(pk->z_C.as<fe>() + (size_t)s * n, p_cur);
        push(pk->z_C.as<fe>() + (size_t)s * n, p_next);
        if (s + 1 < NS) push(pk->z_C.as<fe>() + (size_t)s * n, p_last);
    }
    const uint32_t e_lookup = (uint32_t)pairs.size();
    for (uint32_t l = 0; l < L; ++l) {
        push(pk->zl_C.as<fe>() + (size_t)l * n, p_cur);
        push(pk->zl_C.as<fe>() + (size_t)l * n, p_next);
        push(pk->pa_C.as<fe>() + (size_t)l * n, p_cur);
        push(pk->pa_C.as<fe>() + (size_t)l * n, p_prev);
        push(pk->ps_C.as<fe>() + (size_t)l * n, p_cur);
    }
    const uint32_t n_written = (uint32_t)pairs.size();
    const uint32_t e_h = push(h_poly, p_cur);       // h(x): opened by the multi-open argument, not written
    std::vector<Fr64> evals(pairs.size());
    {
        H2V_TRY(pk->pairs.ensure(pairs.size() * sizeof(EvalPair)));
        H2V_TRY(pk->evals.ensure(pairs.size() * sizeof(fe)));
        H2V_TRY(pk->pts.ensure((points.size() + 8) * sizeof(fe)));
        H2V_TRY(upload(pk, pk->pairs, 0, pairs.data(), pairs.size() * sizeof(EvalPair)));
        H2V_TRY(upload(pk, pk->pts, 0, points.data(), points.size() * sizeof(fe)));
        eval_pairs_kernel<<<(unsigned)pairs.size(), 256, 0, st>>>((const EvalPair *)pk->pairs.p, pk->pts.as<fe>(), (uint32_t)n, pk->evals.as<fe>());
        H2V_LAUNCHED();
        H2V_CU(cudaMemcpyAsync(evals.data(), pk->evals.p, pairs.size() * sizeof(fe), cudaMemcpyDeviceToHost, st));
        H2V_TRY(sync(pk));
    }
    for (uint32_t i = 0; i < n_written; ++i) T.write_scalar(evals[i]);
    lap();   // phase 5: evaluations
    // ---- 13. multi-open argument (SHPLONK)
    // the prover's queries, in upstream's order: advice, permutation products, lookups, fixed, sigma, vanishing
    std::vector<Query> queries;
    {
        size_t e = 0;
        std::vector<Query> adv_q, fix_q, sig_q;
        for (size_t q = 0; q < pk->aq_col.size(); ++q, ++e) adv_q.push_back(Query{pairs[e].poly, pairs[e].point, evals[e]});
        for (size_t q = 0; q < pk->fq_col.size(); ++q, ++e) fix_q.push_back(Query{pairs[e].poly, pairs[e].point, evals[e]});
        ++e;   // random_eval
        for (uint32_t c = 0; c < NP; ++c, ++e) sig_q.push_back(Query{pairs[e].poly, pairs[e].point, evals[e]});
        queries = adv_q;
        // permutation::prover::Evaluated::open: (x, z_s), (wx, z_s) for every set, then (w^last x, z_s) for all but the
        // last set taken in reverse order
        {
            std::vector<uint32_t> at(NS);
            uint32_t pos = e_perm;
            for (uint32_t s = 0; s < NS; ++s) {
                at[s] = pos;
                queries.push_back(Query{pairs[pos].poly, p_cur, evals[pos]});
                queries.push_back(Query{pairs[pos + 1].poly, p_next, evals[pos + 1]});
                pos += (s + 1 < NS) ? 3 : 2;
            }
            for (uint32_t s = NS; s-- > 0;) {
                if (s + 1 == NS) continue;
                queries.push_back(Query{pairs[at[s] + 2].poly, p_last, evals[at[s] + 2]});
            }
        }
        // lookup::prover::Evaluated::open: (x, z), (x, a'), (x, s'), (w^-1 x, a'), (wx, z)
        for (uint32_t l = 0; l < L; ++l) {
            const uint32_t b = e_lookup + 5 * l;
            queries.push_back(Query{pairs[b].poly, p_cur, evals[b]});
            queries.push_back(Query{pairs[b + 2].poly, p_cur, evals[b + 2]});
            queries.push_back(Query{pairs[b + 4].poly, p_cur, evals[b + 4]});
            queries.push_back(Query{pairs[b + 3].poly, p_prev, evals[b + 3]});
            queries.push_back(Query{pairs[b + 1].poly, p_next, evals[b + 1]});
        }
        queries.insert(queries.end(), fix_q.begin(), fix_q.end());
        queries.insert(queries.end(), sig_q.begin(), sig_q.end());
        queries.push_back(Query{h_poly, p_cur, evals[e_h]});
        queries.push_back(Query{pk->rnd_C.as<fe>(), p_cur, evals[e_random]});
    }
    // construct_intermediate_sets: point sets are ordered sets of field elements (BTreeSet<Fr>: numeric order of the
    // canonical values); commitments and rotation sets keep their order of first appearance
    const size_t NPT = points.size();
    std::vector<uint32_t> rank(NPT);      // rank[p] = position of point p in the numeric order
    {
        std::vector<uint32_t> ord(NPT);
        for (size_t i = 0; i < NPT; ++i) ord[i] = (uint32_t)i;
        std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return frh::less_canonical(points[a], points[b]); });
        for (size_t i = 0; i < NPT; ++i) rank[ord[i]] = (uint32_t)i;
    }
    struct Com { const fe *poly; uint64_t mask; };       // mask over ranks
    std::vector<Com> coms;
    std::map<const fe *, size_t> com_of;
    std::map<std::pair<const fe *, uint32_t>, Fr64> eval_of;
    uint64_t super_mask = 0;
    for (const Query &q : queries) {
        const uint64_t bit = (uint64_t)1 << rank[q.pt];
        super_mask |= bit;
        auto it = com_of.find(q.poly);
        if (it == com_of.end()) {
            com_of[q.poly] = coms.size();
            coms.push_back(Com{q.poly, bit});
        } else {
            coms[it->second].mask |= bit;
        }
        eval_of[{q.poly, rank[q.pt]}] = q.eval;
    }
    struct RSet { uint64_t mask; std::vector<const fe *> polys; };
    std::vector<RSet> rsets;
    for (const Com &c : coms) {
        size_t i = 0;
        for (; i < rsets.size(); ++i)
            if (rsets[i].mask == c.mask) break;
        if (i == rsets.size()) rsets.push_back(RSet{c.mask, {}});
        rsets[i].polys.push_back(c.poly);
    }
    std::vector<Fr64> sorted_pts(NPT);
    for (size_t i = 0; i < NPT; ++i) sorted_pts[rank[i]] = points[i];
    auto pts_of = [&](uint64_t mask) {
        std::vector<Fr64> v;
        for (size_t r = 0; r < NPT; ++r)
            if ((mask >> r) & 1) v.push_back(sorted_pts[r]);
        return v;
    };
    const Fr64 ys = T.squeeze_challenge(), vs = T.squeeze_challenge();
    const size_t NR = rsets.size();
    H2V_TRY(pk->sh_S.ensure(NR * n * sizeof(fe)));
    H2V_TRY(pk->sh_A.ensure((n + 8) * sizeof(fe)));
    H2V_TRY(pk->sh_B.ensure(std::max<size_t>(NR, 1) * n * sizeof(fe)));
    size_t max_polys = 0;
    for (auto &rs : rsets) max_polys = std::max(max_polys, rs.polys.size());
    H2V_TRY(pk->ptrs.ensure((max_polys + NR + 8) * sizeof(void *)));
    H2V_TRY(pk->scal.ensure((max_polys + NR + 16) * sizeof(fe)));
    std::vector<std::vector<Fr64>> r_comb(NR);           // sum_j y^j R_ij(X), low degree
    std::vector<std::vector<std::vector<Fr64>>> r_ij(NR);
    fe *Q = pk->sh_B.as<fe>();                                // quotient contributions Q_i, n coefficients each
    for (size_t i = 0; i < NR; ++i) {
        const std::vector<Fr64> ps = pts_of(rsets[i].mask);
        const size_t m = ps.size(), nc = rsets[i].polys.size();
        const std::vector<std::vector<Fr64>> basis = lagrange_basis(ps);
        std::vector<Fr64> ypow(nc);
        Fr64 cur = frh::ONE;
        r_comb[i].assign(m, frh::zero());
        r_ij[i].resize(nc);
        for (size_t j = 0; j < nc; ++j) {
            ypow[j] = cur;
            std::vector<Fr64> ev;
            for (size_t r = 0; r < NPT; ++r)
                if ((rsets[i].mask >> r) & 1) ev.push_back(eval_of[{rsets[i].polys[j], (uint32_t)r}]);
            r_ij[i][j] = lagrange_interpolate(basis, ev);
            for (size_t t = 0; t < m; ++t) r_comb[i][t] = frh::add(r_comb[i][t], frh::mul(r_ij[i][j][t], cur));
            cur = frh::mul(cur, ys);
        }
        // S_i(X) = sum_j y^j P_ij(X)
        H2V_TRY(upload(pk, pk->ptrs, 0, rsets[i].polys.data(), nc * sizeof(void *)));
        H2V_TRY(upload(pk, pk->scal, 0, ypow.data(), nc * sizeof(fe)));
        fe *S = pk->sh_S.as<fe>() + i * n;
        lincomb_kernel<<<gn, 256, 0, st>>>((const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), (uint32_t)nc, (uint32_t)n, S);
        H2V_LAUNCHED();
        // N_i = S_i - sum_j y^j R_ij, then Q_i = N_i / prod (X - p)
        fe *cur_buf = Q + i * n, *oth = pk->sh_A.as<fe>();
        H2V_CU(cudaMemcpyAsync(cur_buf, S, n * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        H2V_TRY(upload(pk, pk->scal, 0, r_comb[i].data(), m * sizeof(fe)));
        sub_low_kernel<<<1, 32, 0, st>>>(cur_buf, pk->scal.as<fe>(), (uint32_t)m);
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        size_t len = n;
        for (size_t t = 0; t < m; ++t) {
            H2V_TRY(h2v_kate_division_dev(cur_buf, len, u64(ps[t]), oth));
            --len;
            std::swap(cur_buf, oth);
        }
        if (cur_buf != Q + i * n) H2V_CU(cudaMemcpyAsync(Q + i * n, cur_buf, len * sizeof(fe), cudaMemcpyDeviceToDevice, st));
        H2V_CU(cudaMemsetAsync(Q + i * n + len, 0, (n - len) * sizeof(fe), st));
        H2V_TRY(sync(pk));
    }
    // h(X) = sum_i v^i Q_i(X)
    {
        std::vector<const fe *> hp(NR);
        std::vector<Fr64> cf(NR);
        Fr64 cur = frh::ONE;
        for (size_t i = 0; i < NR; ++i) {
            hp[i] = Q + i * n;
            cf[i] = cur;
            cur = frh::mul(cur, vs);
        }
        H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), NR * sizeof(void *)));
        H2V_TRY(upload(pk, pk->scal, 0, cf.data(), NR * sizeof(fe)));
        lincomb_kernel<<<gn, 256, 0, st>>>((const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), (uint32_t)NR, (uint32_t)n, hx_dev);
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, hx_dev, 1, pts));
        H2V_TRY(write_points(T, pts));
    }
    const Fr64 uc = T.squeeze_challenge();
    {
        // L(X) = sum_i v^i z_i (S_i(X) - sum_j y^j R_ij(u)) - Z_T(u) h(X);  second opening proof = L / (X - u) / z_0
        const std::vector<Fr64> sup = pts_of(super_mask);
        std::vector<const fe *> hp(NR + 1);
        std::vector<Fr64> cf(NR + 1);
        Fr64 vp = frh::ONE, konst = frh::zero(), z0 = frh::ONE;
        for (size_t i = 0; i < NR; ++i) {
            Fr64 zi = frh::ONE;
            for (size_t r = 0; r < NPT; ++r)
                if (((super_mask & ~rsets[i].mask) >> r) & 1) zi = frh::mul(zi, frh::sub(uc, sorted_pts[r]));
            if (i == 0) z0 = zi;
            Fr64 ri = frh::zero(), yp = frh::ONE;
            for (size_t j = 0; j < rsets[i].polys.size(); ++j) {
                ri = frh::add(ri, frh::mul(yp, eval_small(r_ij[i][j], uc)));
                yp = frh::mul(yp, ys);
            }
            hp[i] = pk->sh_S.as<fe>() + i * n;
            cf[i] = frh::mul(vp, zi);
            konst = frh::add(konst, frh::mul(cf[i], ri));
            vp = frh::mul(vp, vs);
        }
        Fr64 zt = frh::ONE;
        for (const Fr64 &p : sup) zt = frh::mul(zt, frh::sub(uc, p));
        hp[NR] = hx_dev;
        cf[NR] = frh::neg(zt);
        H2V_TRY(upload(pk, pk->ptrs, 0, hp.data(), (NR + 1) * sizeof(void *)));
        H2V_TRY(upload(pk, pk->scal, 0, cf.data(), (NR + 1) * sizeof(fe)));
        fe *Lx = pk->sh_A.as<fe>();
        lincomb_kernel<<<gn, 256, 0, st>>>((const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), (uint32_t)(NR + 1), (uint32_t)n, Lx);
        H2V_LAUNCHED();
        H2V_TRY(upload(pk, pk->scal, 0, &konst, sizeof(fe)));
        sub_low_kernel<<<1, 32, 0, st>>>(Lx, pk->scal.as<fe>(), 1);
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        fe *W = Q;        // the quotient contributions are no longer needed
        H2V_TRY(h2v_kate_division_dev(Lx, n, u64(uc), W));
        H2V_CU(cudaMemsetAsync(W + (n - 1), 0, sizeof(fe), st));
        const Fr64 z0inv = frh::inv(z0);
        H2V_TRY(upload(pk, pk->scal, 0, &z0inv, sizeof(fe)));
        scale_cols_kernel<<<dim3(gn, 1), 256, 0, st>>>(W, (uint32_t)n, pk->scal.as<fe>());
        H2V_LAUNCHED();
        H2V_TRY(sync(pk));
        H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, W, 1, pts));
        H2V_TRY(write_points(T, pts));
    }
    lap();   // phase 6: multi-open argument
    proof.swap(T.out);
    return H2V_OK;
}

}  // namespace

extern "C" {

int h2v_create_proof(h2v_pk_t pk, const uint64_t *const *advice, const uint64_t *const *instances, const uint32_t *instance_len,
                     const uint8_t rng_seed[32], uint8_t *proof_out, size_t proof_cap, size_t *proof_len) {
    if (!pk || !rng_seed || !proof_len) return failf(H2V_EINVAL, "create_proof: NULL argument");
    if ((pk->n_advice && !advice) || (pk->n_instance && (!instances || !instance_len))) return failf(H2V_EINVAL, "create_proof: NULL column list");
    if (cudaSetDevice(pk->dev) != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ECUDA, "create_proof: no CUDA device (libh2v has no CPU fallback)");
    }
    std::lock_guard<std::mutex> lk(pk->mu);
    std::vector<uint8_t> proof;
    int rc = create_proof_locked(pk, advice, instances, instance_len, rng_seed, proof);
    if (rc == H2V_ENOMEM && pk->cached_sigma) {
        // the key's opportunistic cache of extended sigma columns (streamed mode) took memory something else now needs:
        // give it back for good and run the proof again
        cudaStreamSynchronize(pk->st);
        pk->ext_cache.release();
        pk->cached_sigma = 0;
        proof.clear();
        rc = create_proof_locked(pk, advice, instances, instance_len, rng_seed, proof);
    }
    if (rc) {
        cudaStreamSynchronize(pk->st);
        return rc;
    }
    *proof_len = proof.size();
    if (proof.size() > proof_cap || !proof_out) return failf(H2V_EINVAL, "create_proof: proof needs %zu bytes, buffer has %zu", proof.size(), proof_cap);
    memcpy(proof_out, proof.data(), proof.size());
    return H2V_OK;
}
size_t h2v_proof_size(h2v_pk_t pk) {
    if (!pk) return 0;
    const size_t L = pk->lookup_input.size(), NS = pk->n_sets, NP = pk->perm_kind.size();
    const size_t points = pk->n_advice + 2 * L + NS + L + 1 + (pk->degree - 1) + 2;
    const size_t scalars = pk->aq_col.size() + pk->fq_col.size() + 1 + NP + (NS ? 3 * NS - 1 : 0) + 5 * L;
    return 32 * (points + scalars);
}

// ---------------------------------------------------------------- transcript / RNG / hash (host-side ABI)
struct h2v_transcript {
    PoseidonTranscript t;
};
int h2v_transcript_new(h2v_transcript_t *out) {
    if (!out) return failf(H2V_EINVAL, "transcript_new: NULL");
    *out = new h2v_transcript();
    return H2V_OK;
}
void h2v_transcript_free(h2v_transcript_t t) { delete t; }
static affine affine_from(const uint64_t p[8]) {
    affine a;
    memcpy(&a, p, sizeof a);
    return a;
}
int h2v_transcript_common_point(h2v_transcript_t t, const uint64_t affine_pt[8]) {
    if (!t || !affine_pt) return failf(H2V_EINVAL, "transcript: NULL argument");
    if (!t->t.common_point(affine_from(affine_pt))) return failf(H2V_EINVAL, "Cannot write points at infinity to the transcript");
    return H2V_OK;
}
int h2v_transcript_common_scalar(h2v_transcript_t t, const uint64_t s[4]) {
    if (!t || !s) return failf(H2V_EINVAL, "transcript: NULL argument");
    t->t.common_scalar(frh::load(s));
    return H2V_OK;
}
int h2v_transcript_write_point(h2v_transcript_t t, const uint64_t affine_pt[8]) {
    if (!t || !affine_pt) return failf(H2V_EINVAL, "transcript: NULL argument");
    if (!t->t.write_point(affine_from(affine_pt))) return failf(H2V_EINVAL, "Cannot write points at infinity to the transcript");
    return H2V_OK;
}
int h2v_transcript_write_scalar(h2v_transcript_t t, const uint64_t s[4]) {
    if (!t || !s) return failf(H2V_EINVAL, "transcript: NULL argument");
    t->t.write_scalar(frh::load(s));
    return H2V_OK;
}
int h2v_transcript_squeeze_challenge(h2v_transcript_t t, uint64_t out[4]) {
    if (!t || !out) return failf(H2V_EINVAL, "transcript: NULL argument");
    frh::store(out, t->t.squeeze_challenge());
    return H2V_OK;
}
int h2v_transcript_bytes(h2v_transcript_t t, uint8_t *out, size_t cap, size_t *len) {
    if (!t || !len) return failf(H2V_EINVAL, "transcript: NULL argument");
    *len = t->t.out.size();
    if (out && cap >= t->t.out.size()) {
        if (!t->t.out.empty()) memcpy(out, t->t.out.data(), t->t.out.size());
        return H2V_OK;
    }
    return out ? failf(H2V_EINVAL, "transcript_bytes: buffer too small") : H2V_OK;
}
// variant 0: the plain rounds of the Poseidon paper; 1: the sparse form the transcript runs (must agree)
int h2v_poseidon_permutation_variant(uint32_t t, uint32_t r_f, uint32_t r_p, int variant, uint64_t *state);
int h2v_poseidon_permutation(uint32_t t, uint32_t r_f, uint32_t r_p, uint64_t *state) {
    return h2v_poseidon_permutation_variant(t, r_f, r_p, 1, state);
}
int h2v_poseidon_permutation_variant(uint32_t t, uint32_t r_f, uint32_t r_p, int variant, uint64_t *state) {
    if (!state) return failf(H2V_EINVAL, "poseidon_permutation: NULL state");
    if (r_f < 2 || (r_f & 1) || r_f > 64 || r_p > 512) return failf(H2V_EINVAL, "poseidon_permutation: bad round numbers");
    if (t == 3) {
        PoseidonSpec<3> sp = poseidon_make_spec<3>((int)r_f, (int)r_p);
        Fr64 st3[3];
        for (int i = 0; i < 3; ++i) st3[i] = frh::load(state + 4 * i);
        if (variant) poseidon_permute<3>(sp, st3); else poseidon_permute_plain<3>(sp, st3);
        for (int i = 0; i < 3; ++i) frh::store(state + 4 * i, st3[i]);
        return H2V_OK;
    }
    if (t == 5) {
        PoseidonSpec<5> sp = poseidon_make_spec<5>((int)r_f, (int)r_p);
        Fr64 st5[5];
        for (int i = 0; i < 5; ++i) st5[i] = frh::load(state + 4 * i);
        if (variant) poseidon_permute<5>(sp, st5); else poseidon_permute_plain<5>(sp, st5);
        for (int i = 0; i < 5; ++i) frh::store(state + 4 * i, st5[i]);
        return H2V_OK;
    }
    return failf(H2V_EINVAL, "poseidon_permutation: width %u unsupported (3 or 5)", t);
}
int h2v_chacha20_fr_random(const uint8_t seed[32], size_t n, uint64_t *out) {
    if (!seed || (n && !out)) return failf(H2V_EINVAL, "chacha20_fr_random: NULL argument");
    ChaCha20Rng rng(seed);
    for (size_t i = 0; i < n; ++i) frh::store(out + 4 * i, rng.fr_random());
    return H2V_OK;
}
// ---------------------------------------------------------------- gen_srs: seeded setup and the .srs file
// [UPSTREAM] halo2-base utils/fs.rs gen_srs(k): read $PARAMS_DIR/kzg_bn254_{k}.srs, else
// ParamsKZG::setup(k, ChaCha20Rng::from_seed([0; 32])) and write it (scaffold mod.rs:260-261).
int h2v_g2_mul_generator(const uint64_t s_mont[4], uint64_t out[16]) {
    if (!s_mont || !out) return failf(H2V_EINVAL, "g2_mul_generator: NULL argument");
    const Fr64 sc = frh::from_mont(frh::load(s_mont));
    g2h::affine2 r = g2h::mul(g2h::generator(), frh::to_fe(sc));
    memcpy(out, &r, 128);
    return H2V_OK;
}
int h2v_srs_gen(uint32_t k, const uint8_t seed[32], uint64_t *g_out, uint64_t *g_lagrange_out, uint64_t g2_out[16], uint64_t s_g2_out[16]) {
    if (!seed) return failf(H2V_EINVAL, "srs_gen: NULL seed");
    ChaCha20Rng rng(seed);
    const Fr64 s = rng.fr_random();                       // `let s = <E::Scalar>::random(rng);`
    if (g_out || g_lagrange_out) H2V_TRY(h2v_srs_setup(k, s.l, g_out, g_lagrange_out));
    if (g2_out) {
        g2h::affine2 g = g2h::generator();
        memcpy(g2_out, &g, 128);
    }
    if (s_g2_out) H2V_TRY(h2v_g2_mul_generator(s.l, s_g2_out));
    return H2V_OK;
}
// `ParamsKZG::write` (SerdeFormat::RawBytes): k as u32 LE, then g, g_lagrange (2^k G1Affine each: x, y Montgomery limbs,
// 64 bytes), g2, s_g2 (G2Affine: x.c0, x.c1, y.c0, y.c1, 128 bytes)
int h2v_srs_write_file(const char *path, uint32_t k, const uint64_t *g, const uint64_t *g_lagrange, const uint64_t g2[16],
                       const uint64_t s_g2[16]) {
    if (!path || !g || !g_lagrange || !g2 || !s_g2) return failf(H2V_EINVAL, "srs_write_file: NULL argument");
    if (k > 28) return failf(H2V_EINVAL, "srs_write_file: k = %u", k);
    FILE *f = fopen(path, "wb");
    if (!f) return failf(H2V_EINVAL, "srs_write_file: cannot open %s", path);
    const size_t n = (size_t)1 << k;
    bool ok = fwrite(&k, 4, 1, f) == 1 && fwrite(g, 64, n, f) == n && fwrite(g_lagrange, 64, n, f) == n && fwrite(g2, 128, 1, f) == 1 &&
              fwrite(s_g2, 128, 1, f) == 1;
    ok = (fclose(f) == 0) && ok;
    return ok ? H2V_OK : failf(H2V_EINVAL, "srs_write_file: short write to %s", path);
}
// `ParamsKZG::read`: *k_out always receives the file's k; the bases are read when cap_points >= 2^k (else H2V_EINVAL)
int h2v_srs_read_file(const char *path, uint32_t *k_out, uint64_t *g, uint64_t *g_lagrange, size_t cap_points, uint64_t g2[16],
                      uint64_t s_g2[16]) {
    if (!path || !k_out) return failf(H2V_EINVAL, "srs_read_file: NULL argument");
    FILE *f = fopen(path, "rb");
    if (!f) return failf(H2V_EINVAL, "srs_read_file: cannot open %s", path);
    uint32_t k = 0;
    if (fread(&k, 4, 1, f) != 1 || k > 28) {
        fclose(f);
        return failf(H2V_EINVAL, "srs_read_file: bad header in %s", path);
    }
    *k_out = k;
    const size_t n = (size_t)1 << k;
    if (!g || !g_lagrange || !g2 || !s_g2 || cap_points < n) {
        fclose(f);
        return failf(H2V_EINVAL, "srs_read_file: buffers hold %zu points, the file has 2^%u", cap_points, k);
    }
    bool ok = fread(g, 64, n, f) == n && fread(g_lagrange, 64, n, f) == n && fread(g2, 128, 1, f) == 1 && fread(s_g2, 128, 1, f) == 1;
    fclose(f);
    if (!ok) return failf(H2V_EINVAL, "srs_read_file: %s is truncated", path);
    g2h::affine2 a, b;
    memcpy(&a, g2, 128);
    memcpy(&b, s_g2, 128);
    if (!g2h::is_on_curve(a) || !g2h::is_on_curve(b)) return failf(H2V_EINVAL, "srs_read_file: G2 point not on the curve");
    return H2V_OK;
}
int h2v_chacha20_block(const uint8_t seed[32], uint64_t counter, uint8_t out[64]) {
    if (!seed || !out) return failf(H2V_EINVAL, "chacha20_block: NULL argument");
    uint32_t key[8], blk[16];
    memcpy(key, seed, 32);
    ChaCha20Rng::block(key, counter, blk);
    memcpy(out, blk, 64);
    return H2V_OK;
}

}  // extern "C"
