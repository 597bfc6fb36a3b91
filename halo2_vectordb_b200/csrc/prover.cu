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
#include <memory>
#include <mutex>
#include <string>
#include <thread>
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

// A group of B proofs on one key runs phase by phase: proof p's columns of one kind lie after proof p-1's, and the
// kernels below take the proof on grid.z (grid.y where there is no other dimension) with its challenges from a small
// device array (beta_gamma[2p] = beta, beta_gamma[2p + 1] = gamma of proof p).

// permutation argument, plonk/permutation/prover.rs `Argument::commit`: for proof p (grid.z), set s (grid.y) and row i
//   den[s][i] = prod_{c in set} (v_c[i] + beta sigma_c[i] + gamma),  num[s][i] = prod (v_c[i] + beta delta^c w^i + gamma)
struct PermArgs {
    const fe *const *cols;      // n_cols Lagrange columns in permutation order, per proof (n_cols apart)
    const fe *const *sigma;     // their sigma polynomials, Lagrange (the key's: shared by the proofs)
    const fe *omega_pows;       // w^i
    const fe *delta_start;      // per set: delta^(s * chunk)
    const fe *beta_gamma;       // per proof
    fe delta;
    uint32_t n_cols, chunk, n;
};
__global__ void __launch_bounds__(256) perm_numden_kernel(PermArgs a, fe *num, fe *den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, s = blockIdx.y, p = blockIdx.z;
    if (i >= a.n) return;
    const fe *const *cols = a.cols + (size_t)p * a.n_cols;
    const fe beta = ld(a.beta_gamma + 2 * p), gamma = ld(a.beta_gamma + 2 * p + 1);
    const uint32_t c0 = s * a.chunk, c1 = min(c0 + a.chunk, a.n_cols);
    fe cur = fe_mul<Fr>(fe_mul<Fr>(beta, ld(a.omega_pows + i)), ld(a.delta_start + s));
    fe nu = fe_one<Fr>(), de = fe_one<Fr>();
    for (uint32_t c = c0; c < c1; ++c) {
        const fe v = fe_add<Fr>(ld(cols[c] + i), gamma);
        de = fe_mul<Fr>(de, fe_add<Fr>(v, fe_mul<Fr>(beta, ld(a.sigma[c] + i))));
        nu = fe_mul<Fr>(nu, fe_add<Fr>(v, cur));
        cur = fe_mul<Fr>(cur, a.delta);
    }
    const size_t o = ((size_t)p * gridDim.y + s) * a.n + i;
    st(num + o, nu);
    st(den + o, de);
}
// lookup argument, plonk/lookup/prover.rs `Permuted::commit_product`: for proof p (grid.z), lookup l (grid.y) and row i
//   den = (a'[i] + beta)(s'[i] + gamma),  num = (a[i] + beta)(t[i] + gamma)
// inputs: per proof (L apart), tables: the key's; perm_in / perm_tab / num / den: column p * L + l
__global__ void __launch_bounds__(256) lookup_numden_kernel(const fe *const *inputs, const fe *const *tables, const fe *perm_in,
                                                            const fe *perm_tab, const fe *beta_gamma, uint32_t n, fe *num, fe *den) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y, p = blockIdx.z;
    if (i >= n) return;
    const uint32_t col = p * gridDim.y + l;
    const fe beta = ld(beta_gamma + 2 * p), gamma = ld(beta_gamma + 2 * p + 1);
    const size_t o = (size_t)col * n + i;
    st(num + o, fe_mul<Fr>(fe_add<Fr>(ld(inputs[col] + i), beta), fe_add<Fr>(ld(tables[l] + i), gamma)));
    st(den + o, fe_mul<Fr>(fe_add<Fr>(ld(perm_in + o), beta), fe_add<Fr>(ld(perm_tab + o), gamma)));
}
// cols[c][i] *= scalars[c]   (n_cols contiguous columns of n)
__global__ void __launch_bounds__(256) scale_cols_kernel(fe *cols, uint32_t n, const fe *scalars) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe *p = cols + (size_t)blockIdx.y * n + i;
    st(p, fe_mul<Fr>(ld(p), ld(scalars + blockIdx.y)));
}
// job j (grid.y): out[j * out_stride + i] = sum_{t in [off[j], off[j+1])} coef[t] * cols[t][i]
__global__ void __launch_bounds__(256) lincomb_kernel(const fe *const *cols, const fe *coef, const uint32_t *off, uint32_t n, fe *out,
                                                     size_t out_stride) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t t0 = off[blockIdx.y], t1 = off[blockIdx.y + 1];
    fe acc = fe_zero();
    for (uint32_t t = t0; t < t1; ++t) acc = fe_add<Fr>(acc, fe_mul<Fr>(ld(cols[t] + i), ld(coef + t)));
    st(out + (size_t)blockIdx.y * out_stride + i, acc);
}
// job j (grid.x): a[j * stride + i] -= low[j * cnt + i], i < cnt   (subtracting a low-degree polynomial; a job with fewer
// coefficients pads them with zeros, which leave a unchanged)
__global__ void sub_low_kernel(fe *a, size_t stride, const fe *low, uint32_t cnt) {
    fe *aj = a + (size_t)blockIdx.x * stride;
    for (uint32_t i = threadIdx.x; i < cnt; i += blockDim.x) st(aj + i, fe_sub<Fr>(ld(aj + i), ld(low + (size_t)blockIdx.x * cnt + i)));
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
// proof p (grid.y) draws from its own key and block counter into out + p * n
struct ChaChaStream {
    ChaChaKey key;
    uint64_t counter0;
};
__global__ void __launch_bounds__(256) chacha_fr_kernel(const ChaChaStream *streams, uint32_t n, fe *out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const ChaChaKey key = streams[blockIdx.y].key;
    const uint64_t ctr = streams[blockIdx.y].counter0 + i;
    out += (size_t)blockIdx.y * n;
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
    // workspace of a group of proofs (B times what one proof needs), kept between calls; listed by workspace()
    DevBuf adv_L, adv_C, adv_E, inst_L, inst_C, inst_E, pa_L, ps_L, pa_C, ps_C, pa_E, ps_E, z_L, z_C, z_E, zl_L, zl_C, zl_E;
    DevBuf num, den, ptrs, scal, offs, streams, pts, rnd_C, hq, hx_pieces, evals, pairs, sh_S, sh_A, sh_B, sh_T, sh_h, commits;
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
    h2v::MockKey *mock = nullptr;   // the mock prover's key tables, built by the first h2v_pk_mock_prover call
    cudaStream_t st = nullptr;
    int dev = 0;                 // the proof runs on the primary device (columns and key resident there)
    std::mutex mu;
    double last_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // wall-clock per phase of the last call, summed over its groups
};

namespace {

int set_device(int dev, const char *who) {
    if (cudaSetDevice(dev) == cudaSuccess) return H2V_OK;
    cudaGetLastError();
    return failf(H2V_ECUDA, "%s: no CUDA device (libh2v has no CPU fallback)", who);
}
int sync(h2v_pk *pk) {
    H2V_CU(cudaStreamSynchronize(pk->st));
    return H2V_OK;
}
// upload a host array of device pointers / scalars into a (reused) device buffer at byte offset `off`
int upload(h2v_pk *pk, DevBuf &b, size_t off, const void *src, size_t bytes) {
    H2V_CU(cudaMemcpyAsync((char *)b.p + off, src, bytes, cudaMemcpyHostToDevice, pk->st));
    return sync(pk);      // the host staging vectors are short-lived
}
// rows [row0, row0 + rows) of `n_cols` contiguous columns of n <- tails (n_cols x rows, host)
int write_rows(h2v_pk *pk, fe *cols, size_t n, size_t row0, size_t rows, size_t n_cols, const std::vector<Fr64> &tails) {
    if (!rows || !n_cols) return H2V_OK;
    H2V_CU(cudaMemcpy2DAsync(cols + row0, n * sizeof(fe), tails.data(), rows * sizeof(fe), rows * sizeof(fe), n_cols,
                             cudaMemcpyHostToDevice, pk->st));
    return sync(pk);
}
int commit_dev(h2v_pk *pk, int basis, const fe *cols, size_t n_cols, std::vector<affine> &out) {
    out.resize(n_cols);
    if (!n_cols) return H2V_OK;
    H2V_TRY(pk->commits.ensure(n_cols * sizeof(affine)));
    H2V_TRY(h2v_commit_batch_dev(pk->srs, basis, cols, pk->n, n_cols, pk->n, pk->commits.p));
    H2V_CU(cudaMemcpy(out.data(), pk->commits.p, n_cols * sizeof(affine), cudaMemcpyDeviceToHost));
    return H2V_OK;
}
double now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
// The per-proof workspace; a group of B proofs holds B times the buffers of one.
DevBuf *workspace(h2v_pk *pk, size_t i) {
    DevBuf *all[] = {&pk->adv_L, &pk->adv_C, &pk->adv_E, &pk->inst_L, &pk->inst_C, &pk->inst_E, &pk->pa_L, &pk->ps_L, &pk->pa_C, &pk->ps_C,
                     &pk->pa_E, &pk->ps_E, &pk->z_L, &pk->z_C, &pk->z_E, &pk->zl_L, &pk->zl_C, &pk->zl_E, &pk->num, &pk->den,
                     &pk->ptrs, &pk->scal, &pk->offs, &pk->streams, &pk->pts, &pk->rnd_C, &pk->hq, &pk->hx_pieces,
                     &pk->evals, &pk->pairs, &pk->sh_S, &pk->sh_A, &pk->sh_B, &pk->sh_T, &pk->sh_h, &pk->commits};
    return i < sizeof all / sizeof all[0] ? all[i] : nullptr;
}

}  // namespace

namespace h2v {
int check_circuit(const h2v_circuit_t *cs, bool have_column_lists, const char *who) {
    if (cs->degree < 3 || cs->degree > 9) return failf(H2V_EINVAL, "%s: cs.degree() = %u unsupported", who, cs->degree);
    if (cs->k < 2 || cs->k > 24) return failf(H2V_EINVAL, "%s: k = %u unsupported", who, cs->k);
    const size_t n = (size_t)1 << cs->k;
    if ((size_t)cs->blinding_factors + 2 >= n) return failf(H2V_EINVAL, "%s: blinding_factors too large for k", who);
    if (!have_column_lists) return failf(H2V_EINVAL, "%s: NULL column list", who);
    for (uint32_t j = 0; j < cs->n_gates; ++j)
        if (cs->gate_advice[j] >= cs->n_advice || cs->gate_selector[j] >= cs->n_fixed) return failf(H2V_EINVAL, "%s: gate %u out of range", who, j);
    for (uint32_t j = 0; j < cs->n_lookups; ++j)
        if (cs->lookup_input[j] >= cs->n_advice || cs->lookup_table[j] >= cs->n_fixed) return failf(H2V_EINVAL, "%s: lookup %u out of range", who, j);
    for (uint32_t j = 0; j < cs->n_perm; ++j) {
        const uint32_t lim = cs->perm_kind[j] == 0 ? cs->n_advice : cs->perm_kind[j] == 1 ? cs->n_fixed : cs->n_instance;
        if (cs->perm_kind[j] > 2 || cs->perm_index[j] >= lim) return failf(H2V_EINVAL, "%s: permutation column %u out of range", who, j);
    }
    for (uint32_t j = 0; j < cs->n_advice_queries; ++j)
        if (cs->advice_query_col[j] >= cs->n_advice) return failf(H2V_EINVAL, "%s: advice query %u out of range", who, j);
    for (uint32_t j = 0; j < cs->n_fixed_queries; ++j)
        if (cs->fixed_query_col[j] >= cs->n_fixed) return failf(H2V_EINVAL, "%s: fixed query %u out of range", who, j);
    return H2V_OK;
}
size_t group_size_free(size_t n_items, size_t item_bytes, size_t cap, size_t held) {
    cap = std::max<size_t>(1, std::min(cap, n_items));
    if (const char *e = getenv("H2V_PROOF_GROUP")) {
        const long g = atol(e);
        if (g > 0) return std::min<size_t>((size_t)g, cap);
    }
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const size_t margin = (size_t)8 << 30, avail = free_b + held;
    const size_t fit = avail > margin ? (avail - margin) / item_bytes : 1;
    return std::max<size_t>(1, std::min(fit, cap));
}
}  // namespace h2v

extern "C" {

void h2v_pk_free(h2v_pk_t pk) {
    if (!pk) return;
    cudaSetDevice(pk->dev);
    for (DevBuf *b : {&pk->fixed_L, &pk->fixed_C, &pk->fixed_E, &pk->sigma_L, &pk->sigma_C, &pk->sigma_E, &pk->lrows_E, &pk->omega_pows, &pk->scr_E,
                      &pk->ext_cache}) b->release();
    for (size_t i = 0; DevBuf *b = workspace(pk, i); ++i) b->release();
    mock_key_free(pk->mock);
    if (pk->dom) h2v_domain_free(pk->dom);
    if (pk->st) cudaStreamDestroy(pk->st);
    delete pk;
}

int h2v_pk_load(h2v_srs_t srs, const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma,
                const uint64_t vk_transcript_repr[4], h2v_pk_t *out) {
    if (!out) return failf(H2V_EINVAL, "pk_load: out is NULL");
    *out = nullptr;
    if (!srs || !cs || !vk_transcript_repr) return failf(H2V_EINVAL, "pk_load: NULL argument");
    H2V_TRY(check_circuit(cs, !(cs->n_fixed && !fixed) && !(cs->n_perm && !sigma), "pk_load"));
    const size_t n = (size_t)1 << cs->k;
    uint32_t srs_c = 0;
    H2V_TRY(h2v_srs_info(srs, &srs_c, nullptr));

    H2V_TRY(set_device(current_device(), "pk_load"));
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

// ================================================================== create_proof over a group of proofs
namespace {

// the arguments of one h2v_create_proof
struct ProofIn {
    const uint64_t *const *advice;
    const uint64_t *const *instances;
    const uint32_t *instance_len;
    const uint8_t *seed;
};
// The advice and instances of a group's proofs generated on the device by a witness program
// (h2v_create_proofs_from_inputs): proof p of the group has the inputs at inputs + p n_inputs 4, and its instances are
// downloaded to instances + p n_instances 4, where the proof's ProofIn.instances points
struct Generated {
    h2v_witness_program *prog;
    size_t n_inputs, n_instances;
    const uint64_t *inputs;
    uint64_t *instances;
    Generated at(size_t p) const { return {prog, n_inputs, n_instances, inputs + p * n_inputs * 4, instances + p * n_instances * 4}; }
};
// what one proof of a group carries from phase to phase: its own RNG, transcript and challenges
struct ProofState {
    PoseidonTranscript T;
    ChaCha20Rng rng;
    Fr64 beta, gamma, y, x, xn, ys, vs, uc;
    explicit ProofState(const uint8_t *seed) : rng(seed) {}
};

enum ColForm { LAGRANGE, COEFF, EXTENDED };

// What the phases of one group of proofs share.  Proofs in[0 .. B) run in lockstep: every commit, transform, grand
// product and column kernel of a phase is one call over the B proofs' columns (proof p's columns of a kind after proof
// p - 1's), while each proof keeps its own RNG (upstream's draw order) and transcript (its own challenges) in P[p].
struct Group {
    h2v_pk *pk;
    size_t B;
    const ProofIn *in;
    const Generated *gen;                           // NULL: in[p].advice and in[p].instances are host columns
    std::vector<std::unique_ptr<ProofState>> P;
    size_t n, ne;
    uint32_t A, F, I, L, G, NP, NS, NH, bf, u;      // NH: quotient pieces of n coefficients each
    unsigned gn;                                    // blocks of 256 rows
    size_t &bad;                                    // on a failure traced to one proof, that proof (else SIZE_MAX)
    std::vector<affine> pts;                        // commitments of the current step
    fe *pieces = nullptr;                           // the B x NH quotient pieces, contiguous columns of n (commit_quotient)
    double t_phase = now_ms();
    int phase = 0;

    Group(h2v_pk *pk_, size_t B_, const ProofIn *in_, const Generated *gen_, size_t &bad_)
        : pk(pk_), B(B_), in(in_), gen(gen_), n(pk_->n), ne(pk_->ne), A(pk_->n_advice), F(pk_->n_fixed), I(pk_->n_instance),
          L((uint32_t)pk_->lookup_input.size()), G((uint32_t)pk_->gate_advice.size()), NP((uint32_t)pk_->perm_kind.size()),
          NS(pk_->n_sets), NH(pk_->degree - 1), bf(pk_->bf), u(pk_->u), gn((unsigned)((pk_->n + 255) / 256)), bad(bad_) {
        bad = SIZE_MAX;
        for (size_t p = 0; p < B; ++p) P.emplace_back(new ProofState(in[p].seed));
    }
    // column idx of a kind (0 advice, 1 fixed, 2 instance) of proof p; the fixed columns are the key's, shared by the proofs
    const fe *col(ColForm form, size_t p, uint8_t kind, uint32_t idx) const {
        const DevBuf *bufs[3][3] = {{&pk->adv_L, &pk->adv_C, &pk->adv_E}, {&pk->fixed_L, &pk->fixed_C, &pk->fixed_E},
                                    {&pk->inst_L, &pk->inst_C, &pk->inst_E}};
        const size_t at = kind == 0 ? p * A + idx : kind == 1 ? idx : p * I + idx;
        return bufs[kind][form]->as<fe>() + at * (form == EXTENDED ? ne : n);
    }
    std::vector<Fr64> beta_gamma() const {      // beta, gamma of every proof, as the column kernels read them
        std::vector<Fr64> v;
        for (auto &s : P) v.insert(v.end(), {s->beta, s->gamma});
        return v;
    }
    // ends the current phase of h2v_pk_last_phase_ms
    void lap() {
        const double t = now_ms();
        if (phase < 7) pk->last_ms[phase++] += t - t_phase;
        t_phase = t;
    }
};

// f(p) for every proof p < B, on up to B host threads (the proofs' transcripts and point-set arithmetic are independent).
// h2v_last_error() is per thread: a worker's error text is carried back to the caller's thread.
template <class F> int par_proofs(size_t B, F f) {
    if (B == 1) return f(0);
    const size_t W = std::min<size_t>(B, std::max(1u, std::thread::hardware_concurrency()));
    std::vector<int> rc(B, H2V_OK);
    std::vector<std::string> msg(B);
    std::vector<std::thread> th;
    for (size_t w = 0; w < W; ++w)
        th.emplace_back([&, w] {
            for (size_t p = w; p < B; p += W)
                if ((rc[p] = f(p))) msg[p] = h2v_last_error();
        });
    for (auto &t : th) t.join();
    for (size_t p = 0; p < B; ++p)
        if (rc[p]) return set_error(rc[p], msg[p].c_str());
    return H2V_OK;
}

// the host vector into a device buffer that grows to fit it (the stream is idle when this returns)
template <class T> int put(h2v_pk *pk, DevBuf &b, const std::vector<T> &v) {
    if (v.empty()) return H2V_OK;
    if (v.size() * sizeof(T) > b.cap) H2V_TRY(sync(pk));      // nothing queued may still read the buffer that is replaced
    H2V_TRY(b.ensure(v.size() * sizeof(T)));
    return upload(pk, b, 0, v.data(), v.size() * sizeof(T));
}
// out + j * out_stride = sum_{t in [off[j], off[j+1])} coef[t] * cols[t] over `len` rows, one launch for every job
int lincomb(h2v_pk *pk, const std::vector<const fe *> &cols, const std::vector<Fr64> &coef, const std::vector<uint32_t> &off, fe *out,
            size_t out_stride, size_t len) {
    H2V_TRY(put(pk, pk->ptrs, cols));
    H2V_TRY(put(pk, pk->scal, coef));
    H2V_TRY(put(pk, pk->offs, off));
    lincomb_kernel<<<dim3((unsigned)((len + 255) / 256), (unsigned)(off.size() - 1)), 256, 0, pk->st>>>(
        (const fe *const *)pk->ptrs.p, pk->scal.as<fe>(), pk->offs.as<uint32_t>(), (uint32_t)len, out, out_stride);
    H2V_LAUNCHED();
    return H2V_OK;
}
// a[j * stride + i] -= low[j][i] for every job j (low: the same number of coefficients per job, zero-padded)
int sub_low(h2v_pk *pk, fe *a, size_t stride, const std::vector<Fr64> &low, size_t jobs) {
    const uint32_t cnt = (uint32_t)(low.size() / jobs);
    H2V_TRY(put(pk, pk->scal, low));
    sub_low_kernel<<<(unsigned)jobs, 32, 0, pk->st>>>(a, stride, pk->scal.as<fe>(), cnt);
    H2V_LAUNCHED();
    return H2V_OK;
}
// out + p n = sum_i c^i cols[(p m + i) n] for every proof p, with c = the proof's challenge `c`; one launch
int sum_powers(Group &g, const fe *cols, size_t m, Fr64 ProofState::*c, fe *out) {
    std::vector<const fe *> hp(g.B * m);
    std::vector<Fr64> cf(g.B * m);
    std::vector<uint32_t> off(g.B + 1);
    for (size_t p = 0; p < g.B; ++p) {
        Fr64 cur = frh::ONE;
        off[p] = (uint32_t)(p * m);
        for (size_t i = 0; i < m; ++i) {
            hp[p * m + i] = cols + (p * m + i) * g.n;
            cf[p * m + i] = cur;
            cur = frh::mul(cur, (*g.P[p]).*c);
        }
    }
    off[g.B] = (uint32_t)(g.B * m);
    return lincomb(g.pk, hp, cf, off, out, g.n, g.n);
}
// proof p's commitments pts[p per_proof .. (p + 1) per_proof) into its transcript, for every proof; a point at infinity
// fails the proof it belongs to.  absorb: hash them on the transcripts' worker threads while the next kernels run.
int write_commitments(Group &g, const std::vector<affine> &pts, size_t per_proof, bool absorb) {
    for (size_t p = 0; p < g.B; ++p) {
        for (size_t i = 0; i < per_proof; ++i)
            if (!g.P[p]->T.write_point(pts[p * per_proof + i])) {
                g.bad = p;
                return failf(H2V_EINVAL, "create_proof: Cannot write points at infinity to the transcript");
            }
        if (absorb) g.P[p]->T.absorb_async();
    }
    return H2V_OK;
}
// the end of a grand-product step (permutation/prover.rs commit, lookup/prover.rs commit_product): per proof and
// column, bf random rows at n - bf and one blind; then the columns of z are committed and written
int commit_products(Group &g, DevBuf &z, size_t cols_per_proof) {
    const size_t cols = g.B * cols_per_proof;
    std::vector<Fr64> zt(cols * g.bf);
    for (size_t p = 0; p < g.B; ++p)
        for (size_t c = 0; c < cols_per_proof; ++c) {
            for (uint32_t i = 0; i < g.bf; ++i) zt[(p * cols_per_proof + c) * g.bf + i] = g.P[p]->rng.fr_random();   // rows n - bf .. n - 1
            (void)g.P[p]->rng.fr_random();                                                                        // product blind
        }
    H2V_TRY(write_rows(g.pk, z.as<fe>(), g.n, g.n - g.bf, g.bf, cols, zt));
    H2V_TRY(commit_dev(g.pk, H2V_BASIS_LAGRANGE, z.as<fe>(), cols, g.pts));
    return write_commitments(g, g.pts, cols_per_proof, true);
}

// ---- phase 0.  plonk/prover.rs create_proof steps 1-4: vk and instances into the transcripts (hash_into, common_scalar);
//      the advice columns uploaded (or generated in place), blinded in their last bf + 1 rows and committed
int instances_and_advice(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, BA = B * g.A, BI = B * g.I;
    const uint32_t A = g.A, bf = g.bf;
    for (auto &s : g.P) s->T.common_scalar(pk->vk_repr);
    H2V_TRY(pk->inst_L.ensure(std::max<size_t>(1, BI) * n * sizeof(fe)));
    H2V_TRY(pk->inst_C.ensure(std::max<size_t>(1, BI) * n * sizeof(fe)));
    H2V_TRY(pk->inst_E.ensure(std::max<size_t>(1, BI) * g.ne * sizeof(fe)));
    H2V_TRY(pk->adv_L.ensure(BA * n * sizeof(fe)));
    H2V_TRY(pk->adv_C.ensure(BA * n * sizeof(fe)));
    if (g.gen) {      // the columns straight into adv_L / inst_L; the instances also to the host, for the transcripts
        size_t bad_w = B;
        const int rc = witness_generate_dev(g.gen->prog, pk->st, B, g.gen->inputs, pk->adv_L.as<fe>(), pk->inst_L.as<fe>(), g.I ? n : 0,
                                            g.gen->instances, &bad_w);
        if (bad_w < B) g.bad = bad_w;
        H2V_TRY(rc);
    }
    if (g.I) {
        std::vector<Fr64> inst(g.gen ? 0 : BI * n, frh::zero());
        for (size_t p = 0; p < B; ++p)
            for (uint32_t c = 0; c < g.I; ++c)
                for (uint32_t i = 0; i < g.in[p].instance_len[c]; ++i) {
                    const Fr64 v = frh::load(g.in[p].instances[c] + 4 * i);
                    g.P[p]->T.common_scalar(v);
                    if (!g.gen) inst[(p * g.I + c) * n + i] = v;
                }
        if (!g.gen) H2V_TRY(upload(pk, pk->inst_L, 0, inst.data(), BI * n * sizeof(fe)));
        H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_LAGRANGE_TO_COEFF, pk->inst_L.p, n, pk->inst_C.p, n, BI));
    }
    std::vector<Fr64> tails(BA * (bf + 1));
    std::vector<const uint64_t *> adv(g.gen ? 0 : BA);
    for (size_t p = 0; p < B; ++p) {
        ChaCha20Rng &rng = g.P[p]->rng;
        for (size_t t = 0; t < (size_t)A * (bf + 1); ++t) tails[p * A * (bf + 1) + t] = rng.fr_random();   // column by column, rows u .. n-1
        for (uint32_t c = 0; c < A; ++c) (void)rng.fr_random();          // one Blind per column (unused by KZG, but drawn)
        if (!g.gen)
            for (uint32_t c = 0; c < A; ++c) adv[p * A + c] = g.in[p].advice[c];
    }
    if (g.gen) {      // rows u .. n-1 of the resident columns <- the tails; h2v_commit_batch_dev spreads the commits over the devices
        H2V_TRY(write_rows(pk, pk->adv_L.as<fe>(), n, g.u, bf + 1, BA, tails));
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->adv_L.as<fe>(), BA, g.pts));
    } else {      // each device uploads its block of the B x A columns in sub-batches (the next one crosses while the previous
                  // one is committed), writes the tails, commits the block and leaves it in adv_L
        g.pts.resize(BA);
        H2V_TRY(h2v_commit_batch_resident(pk->srs, H2V_BASIS_LAGRANGE, adv.data(), BA, n, (const uint64_t *)tails.data(), g.u, bf + 1, pk->adv_L.p,
                                          n, (uint64_t *)g.pts.data()));
    }
    return write_commitments(g, g.pts, A, true);      // hashed while the lookup permutations run
}

// ---- phase 1.  lookup/prover.rs commit_permuted (step 5): the permuted input and table columns A', S' of every lookup,
//      blinded and committed.  theta is squeezed at its place in the transcript, just before A' / S' are written:
//      single-expression lookups have nothing to compress, so the permutations do not wait for it
int permuted_lookups(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, L = g.L, BL = B * L;
    const uint32_t bf = g.bf;
    H2V_TRY(pk->pa_L.ensure(std::max<size_t>(1, BL) * n * sizeof(fe)));
    H2V_TRY(pk->ps_L.ensure(std::max<size_t>(1, BL) * n * sizeof(fe)));
    std::vector<affine> written(2 * BL);      // A'_l, S'_l of each lookup of each proof, in transcript order
    if (L) {
        std::vector<const void *> li(BL), lt(BL);
        for (size_t p = 0; p < B; ++p)
            for (uint32_t l = 0; l < L; ++l) {
                li[p * L + l] = g.col(LAGRANGE, p, 0, pk->lookup_input[l]);
                lt[p * L + l] = g.col(LAGRANGE, p, 1, pk->lookup_table[l]);      // the key's table: sorted once for the group
            }
        int rc = h2v_permute_expression_pair_batch_dev(li.data(), lt.data(), BL, g.u, pk->pa_L.as<fe>(), n, pk->ps_L.as<fe>(), n);
        if (rc == H2V_EINVAL && B > 1) {
            // an input value outside its table: find the proof it belongs to
            for (size_t p = 0; p < B; ++p) {
                const int rc_p = h2v_permute_expression_pair_batch_dev(li.data() + p * L, lt.data() + p * L, L, g.u, pk->pa_L.as<fe>(), n,
                                                                       pk->ps_L.as<fe>(), n);
                if (rc_p) {
                    g.bad = p;
                    return rc_p;
                }
            }
        }
        if (rc) return rc;
        std::vector<Fr64> ta(BL * (bf + 1)), ts(BL * (bf + 1));
        for (size_t p = 0; p < B; ++p) {
            ChaCha20Rng &rng = g.P[p]->rng;
            for (uint32_t l = 0; l < L; ++l) {
                const size_t col = p * L + l;
                for (uint32_t i = 0; i <= bf; ++i) ta[col * (bf + 1) + i] = rng.fr_random();
                for (uint32_t i = 0; i <= bf; ++i) ts[col * (bf + 1) + i] = rng.fr_random();
                (void)rng.fr_random();     // permuted input blind
                (void)rng.fr_random();     // permuted table blind
            }
        }
        H2V_TRY(write_rows(pk, pk->pa_L.as<fe>(), n, g.u, bf + 1, BL, ta));
        H2V_TRY(write_rows(pk, pk->ps_L.as<fe>(), n, g.u, bf + 1, BL, ts));
        std::vector<affine> ca, cs;
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->pa_L.as<fe>(), BL, ca));
        H2V_TRY(commit_dev(pk, H2V_BASIS_LAGRANGE, pk->ps_L.as<fe>(), BL, cs));
        for (size_t c = 0; c < BL; ++c) {
            written[2 * c] = ca[c];
            written[2 * c + 1] = cs[c];
        }
    }
    for (auto &s : g.P) (void)s->T.squeeze_challenge();      // theta
    return write_commitments(g, written, 2 * L, false);
}

// ---- phase 2.  permutation/prover.rs Argument::commit (step 6): beta, gamma; the grand product of every permutation set
int permutation_products(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, BS = B * g.NS;
    const uint32_t NP = g.NP, NS = g.NS, L = g.L, u = g.u;
    for (auto &s : g.P) {
        s->beta = s->T.squeeze_challenge();
        s->gamma = s->T.squeeze_challenge();
    }
    H2V_TRY(pk->z_L.ensure(std::max<size_t>(1, BS) * n * sizeof(fe)));
    H2V_TRY(pk->num.ensure(std::max<size_t>(1, B * std::max(NS, L)) * n * sizeof(fe)));
    H2V_TRY(pk->den.ensure(std::max<size_t>(1, B * std::max(NS, L)) * n * sizeof(fe)));
    H2V_TRY(pk->ptrs.ensure((size_t)(4 * (NP + g.G + L) * B + 4096) * sizeof(void *)));
    H2V_TRY(pk->scal.ensure((size_t)(NS + g.A + g.F + NP + 3 * NS + 5 * L + 64) * B * sizeof(fe) + 4096));
    if (!NS) return H2V_OK;
    std::vector<const fe *> hp((B + 1) * NP);
    for (size_t p = 0; p < B; ++p)
        for (uint32_t c = 0; c < NP; ++c) hp[p * NP + c] = g.col(LAGRANGE, p, pk->perm_kind[c], pk->perm_index[c]);
    for (uint32_t c = 0; c < NP; ++c) hp[B * NP + c] = pk->sigma_L.as<fe>() + (size_t)c * n;
    H2V_TRY(put(pk, pk->ptrs, hp));
    std::vector<Fr64> sc(NS);                       // delta^(s * chunk), then beta, gamma of every proof
    const Fr64 dchunk = frh::pow_u64(pk->delta, pk->chunk);
    Fr64 cur = frh::ONE;
    for (uint32_t s = 0; s < NS; ++s) {
        sc[s] = cur;
        cur = frh::mul(cur, dchunk);
    }
    for (const Fr64 &v : g.beta_gamma()) sc.push_back(v);
    H2V_TRY(put(pk, pk->scal, sc));
    PermArgs pa;
    pa.cols = (const fe *const *)pk->ptrs.p;
    pa.sigma = pa.cols + B * NP;
    pa.omega_pows = pk->omega_pows.as<fe>();
    pa.delta_start = pk->scal.as<fe>();
    pa.beta_gamma = pk->scal.as<fe>() + NS;
    pa.delta = frh::to_fe(pk->delta);
    pa.n_cols = NP; pa.chunk = pk->chunk; pa.n = (uint32_t)n;
    perm_numden_kernel<<<dim3(g.gn, NS, (unsigned)B), 256, 0, pk->st>>>(pa, pk->num.as<fe>(), pk->den.as<fe>());
    H2V_LAUNCHED();
    H2V_TRY(sync(pk));
    // z_s with z_s[0] = 1; then chain: z_s *= z_{s-1}[u] (upstream carries `last_z` from set to set)
    H2V_TRY(h2v_grand_product_dev(pk->num.p, pk->den.p, n, BS, pk->z_L.p));
    std::vector<Fr64> last(BS), scale(BS);
    H2V_CU(cudaMemcpy2D(last.data(), sizeof(fe), pk->z_L.as<fe>() + u, n * sizeof(fe), sizeof(fe), BS, cudaMemcpyDeviceToHost));
    for (size_t p = 0; p < B; ++p) {
        cur = frh::ONE;
        for (uint32_t s = 0; s < NS; ++s) {
            scale[p * NS + s] = cur;
            cur = frh::mul(cur, last[p * NS + s]);
        }
    }
    H2V_TRY(put(pk, pk->scal, scale));
    scale_cols_kernel<<<dim3(g.gn, (unsigned)BS), 256, 0, pk->st>>>(pk->z_L.as<fe>(), (uint32_t)n, pk->scal.as<fe>());
    H2V_LAUNCHED();
    return commit_products(g, pk->z_L, NS);      // hashed while the lookup products are built and committed
}

//      lookup/prover.rs Permuted::commit_product (step 7): the grand product of every lookup
int lookup_products(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, L = g.L, BL = B * L;
    H2V_TRY(pk->zl_L.ensure(std::max<size_t>(1, BL) * n * sizeof(fe)));
    if (!L) return H2V_OK;
    std::vector<const fe *> hp(BL + L);
    for (size_t p = 0; p < B; ++p)
        for (uint32_t l = 0; l < L; ++l) hp[p * L + l] = g.col(LAGRANGE, p, 0, pk->lookup_input[l]);
    for (uint32_t l = 0; l < L; ++l) hp[BL + l] = g.col(LAGRANGE, 0, 1, pk->lookup_table[l]);
    H2V_TRY(put(pk, pk->ptrs, hp));
    H2V_TRY(put(pk, pk->scal, g.beta_gamma()));
    lookup_numden_kernel<<<dim3(g.gn, (unsigned)L, (unsigned)B), 256, 0, pk->st>>>((const fe *const *)pk->ptrs.p, (const fe *const *)pk->ptrs.p + BL,
                                                                                 pk->pa_L.as<fe>(), pk->ps_L.as<fe>(), pk->scal.as<fe>(), (uint32_t)n,
                                                                                 pk->num.as<fe>(), pk->den.as<fe>());
    H2V_LAUNCHED();
    H2V_TRY(sync(pk));
    H2V_TRY(h2v_grand_product_dev(pk->num.p, pk->den.p, n, BL, pk->zl_L.p));
    return commit_products(g, pk->zl_L, L);
}

// ---- phase 3.  vanishing/prover.rs Argument::commit (step 8): the random polynomial, n consecutive Fr::random draws =
//      n consecutive key-stream blocks, produced on the device, every proof's in one launch
int random_polynomial(Group &g) {
    h2v_pk *pk = g.pk;
    H2V_TRY(pk->rnd_C.ensure(g.B * g.n * sizeof(fe)));
    std::vector<ChaChaStream> cs(g.B);
    for (size_t p = 0; p < g.B; ++p) {
        ChaCha20Rng &rng = g.P[p]->rng;
        memcpy(cs[p].key.k, rng.key, 32);
        cs[p].counter0 = rng.next_block();
        rng.skip_fr(g.n);
        (void)rng.fr_random();      // random_blind
    }
    H2V_TRY(put(pk, pk->streams, cs));
    chacha_fr_kernel<<<dim3(g.gn, (unsigned)g.B), 256, 0, pk->st>>>(pk->streams.as<ChaChaStream>(), (uint32_t)g.n, pk->rnd_C.as<fe>());
    H2V_LAUNCHED();
    H2V_TRY(sync(pk));
    H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, pk->rnd_C.as<fe>(), g.B, g.pts));
    return write_commitments(g, g.pts, 1, true);
}

//      plonk/prover.rs create_proof, the polynomials of steps 9-11: coefficient and extended forms of the proof's columns
//      (no challenge involved: they run while the commitments above are hashed).  A streamed key keeps no extended
//      advice columns: evaluate_h_streamed rebuilds them slice by slice.
int transform_columns(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t n = g.n, ne = g.ne, BA = g.B * g.A, BI = g.B * g.I, BL = g.B * g.L, BS = g.B * g.NS;
    const int L2C = H2V_OP_LAGRANGE_TO_COEFF, C2E = H2V_OP_COEFF_TO_EXTENDED;
    const bool stream = pk->stream_ext;      // (a streamed key proves in groups of one)
    // (the per-proof buffers are kept between proofs, also in streamed mode: with peer access enabled, freeing and
    // re-allocating gigabytes every proof costs more than the transforms themselves -- measured on two devices)
    if (!stream) H2V_TRY(pk->adv_E.ensure(BA * ne * sizeof(fe)));
    H2V_TRY(h2v_domain_transform_dev(pk->dom, L2C, pk->adv_L.p, n, pk->adv_C.p, n, BA));
    if (!stream) H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, pk->adv_C.p, n, pk->adv_E.p, ne, BA));
    if (g.I) H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, pk->inst_C.p, n, pk->inst_E.p, ne, BI));
    struct Tr { DevBuf *Lb, *Cb, *Eb; size_t cnt; } trs[4] = {{&pk->pa_L, &pk->pa_C, &pk->pa_E, BL}, {&pk->ps_L, &pk->ps_C, &pk->ps_E, BL},
                                                            {&pk->z_L, &pk->z_C, &pk->z_E, BS}, {&pk->zl_L, &pk->zl_C, &pk->zl_E, BL}};
    for (auto &t : trs) {
        H2V_TRY(t.Cb->ensure(std::max<size_t>(1, t.cnt) * n * sizeof(fe)));
        H2V_TRY(t.Eb->ensure(std::max<size_t>(1, t.cnt) * ne * sizeof(fe)));
        if (!t.cnt) continue;
        H2V_TRY(h2v_domain_transform_dev(pk->dom, L2C, t.Lb->p, n, t.Cb->p, n, t.cnt));
        H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, t.Cb->p, n, t.Eb->p, ne, t.cnt));
    }
    return H2V_OK;
}

// ---- phase 4.  plonk/evaluation.rs Evaluator::evaluate_h over resident extended columns: the gate, permutation and
//      lookup folds of every proof into h (proof p's at h + p ne), three launches through one pointer table
int evaluate_h_resident(Group &g, fe *h) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, ne = g.ne;
    const uint32_t G = g.G, NP = g.NP, L = g.L;
    const size_t per = 2 * (size_t)G + 2 * (size_t)NP;
    std::vector<const fe *> hp(B * per);
    for (size_t p = 0; p < B; ++p) {
        const fe **t = hp.data() + p * per;
        for (uint32_t j = 0; j < G; ++j) {
            t[j] = g.col(EXTENDED, p, 1, pk->gate_selector[j]);
            t[G + j] = g.col(EXTENDED, p, 0, pk->gate_advice[j]);
        }
        for (uint32_t c = 0; c < NP; ++c) {
            t[2 * G + c] = g.col(EXTENDED, p, pk->perm_kind[c], pk->perm_index[c]);
            t[2 * G + NP + c] = pk->sigma_E.as<fe>() + (size_t)c * ne;
        }
    }
    // the lookups' five columns per lookup after the gate and permutation tables; every proof's y, beta, gamma
    for (size_t p = 0; p < B; ++p)
        for (uint32_t l = 0; l < L; ++l) {
            const size_t col = p * L + l;
            const fe *five[5] = {g.col(EXTENDED, p, 0, pk->lookup_input[l]), g.col(EXTENDED, p, 1, pk->lookup_table[l]), pk->pa_E.as<fe>() + col * ne,
                                 pk->ps_E.as<fe>() + col * ne, pk->zl_E.as<fe>() + col * ne};
            hp.insert(hp.end(), five, five + 5);
        }
    H2V_TRY(put(pk, pk->ptrs, hp));
    std::vector<Fr64> ybg;
    for (auto &s : g.P) ybg.insert(ybg.end(), {s->y, s->beta, s->gamma});
    H2V_TRY(put(pk, pk->scal, ybg));
    const void *const *tab = (const void *const *)pk->ptrs.p;
    const fe *l0 = pk->lrows_E.as<fe>();
    QuotientBatch qb;
    qb.h = h; qb.h_stride = ne; qb.scal = pk->scal.p; qb.n_proofs = B;
    qb.n_gates = G; qb.gate_tab = tab; qb.gate_pstride = per;
    qb.n_perm = NP; qb.chunk = pk->chunk; qb.perm_tab = tab + 2 * G; qb.perm_pstride = per;
    qb.z = pk->z_E.p; qb.z_stride = ne; qb.z_pstride = (size_t)g.NS * ne; qb.blinding_factors = g.bf;
    qb.n_lookups = L; qb.lookup_tab = tab + B * per; qb.lookup_pstride = 5 * (size_t)L;
    qb.l0 = l0; qb.l_last = l0 + ne; qb.l_active = l0 + 2 * ne;
    return quotient_batch_dev(pk->dom, qb);
}

// Once per streamed key: what is left of the device's memory after the first proof's buffers exist keeps the extended forms
// of the first sigma polynomials (H2V_EXT_CACHE_COLS of them if set, else as many as leave 8 GB free)
int fill_sigma_cache(Group &g) {
    h2v_pk *pk = g.pk;
    if (pk->cache_tried) return H2V_OK;
    pk->cache_tried = true;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const char *e = getenv("H2V_EXT_CACHE_COLS");
    const size_t margin = (size_t)8 << 30;
    size_t want = e ? (size_t)atoi(e) : (free_b > margin ? (free_b - margin) / (g.ne * sizeof(fe)) : 0);
    want = std::min<size_t>(want, g.NP);
    if (want >= (e ? 1u : 8u) && pk->ext_cache.ensure(want * g.ne * sizeof(fe)) == H2V_OK) {
        H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_COEFF_TO_EXTENDED, pk->sigma_C.p, g.n, pk->ext_cache.p, g.ne, want));
        pk->cached_sigma = want;
    }
    return H2V_OK;
}

//      plonk/evaluation.rs Evaluator::evaluate_h for a streamed key (one proof): the same folds, in upstream's order, over
//      slices of columns whose extended forms are rebuilt into `scr_E` from the resident coefficient forms (every term
//      reads columns of its own gate / set / lookup only).  hp_acc: ne elements free until the division.
int evaluate_h_streamed(Group &g, fe *h_ext, fe *hp_acc) {
    h2v_pk *pk = g.pk;
    const size_t n = g.n, ne = g.ne, SC = pk->scr_cols;
    const uint32_t A = g.A, G = g.G, NP = g.NP, NS = g.NS, L = g.L, bf = g.bf;
    const int C2E = H2V_OP_COEFF_TO_EXTENDED;
    const Fr64 &y = g.P[0]->y, &beta = g.P[0]->beta, &gamma = g.P[0]->gamma;
    const fe *l0 = pk->lrows_E.as<fe>(), *ll = l0 + ne, *la = l0 + 2 * ne;
    H2V_TRY(pk->scr_E.ensure(SC * ne * sizeof(fe)));
    fe *scr = pk->scr_E.as<fe>();
    // coeff_to_extended of a list of coefficient columns into consecutive scratch slots; neighbours share one launch
    const bool timing = getenv("H2V_PROVE_TIMING") != nullptr;
    double t_ext = 0, t_fold = 0, t_mark = now_ms();
    auto mark = [&](double &acc) {
        if (!timing) return;
        cudaDeviceSynchronize();
        const double t = now_ms();
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
    // slices serves both folds -- the gates into h, the permutation into a second accumulator hp_acc, joined as
    // h <- h y^(permutation terms) + hp_acc.  Each advice column is then extended once instead of twice.  Any other
    // constraint system takes the two separate loops below.
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
        H2V_CU(cudaMemsetAsync(hp_acc, 0, ne * sizeof(fe), pk->st));
        H2V_TRY(sync(pk));
        H2V_TRY(fill_sigma_cache(g));
        const size_t BS = std::max<size_t>(1, SC / (3 * (size_t)pk->chunk));
        std::vector<const fe *> pc, sg, gq, ga;
        for (size_t s0 = 0; s0 < NS; s0 += BS) {
            const size_t s1 = std::min<size_t>(NS, s0 + BS), c0 = s0 * pk->chunk, c1 = std::min<size_t>(NP, s1 * pk->chunk), cnt = c1 - c0;
            src.clear(); pc.clear(); sg.clear(); gq.clear(); ga.clear();
            size_t slot = 0;
            for (size_t c = c0; c < c1; ++c) {
                src.push_back(g.col(COEFF, 0, pk->perm_kind[c], pk->perm_index[c]));
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
                src.push_back(g.col(COEFF, 0, 1, pk->gate_selector[gate_of_adv[pk->perm_index[c]]]));
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
        // h <- h y^T + hp_acc, T = the permutation argument's terms: 2 + (NS - 1) + NS
        H2V_TRY(lincomb(pk, {h_ext, hp_acc}, {frh::pow_u64(y, 2ull * NS + 1), frh::ONE}, {0, 2}, h_ext, ne, ne));
        H2V_TRY(sync(pk));
        mark(t_fold);
    } else {
        const size_t BG = SC / 2;
        for (size_t g0 = 0; g0 < G; g0 += BG) {
            const size_t b = std::min<size_t>(BG, G - g0);
            src.clear();
            hp.assign(2 * b, nullptr);
            for (size_t j = 0; j < b; ++j) src.push_back(g.col(COEFF, 0, 1, pk->gate_selector[g0 + j]));
            for (size_t j = 0; j < b; ++j) src.push_back(g.col(COEFF, 0, 0, pk->gate_advice[g0 + j]));
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
            for (size_t c = c0; c < c1; ++c) src.push_back(g.col(COEFF, 0, pk->perm_kind[c], pk->perm_index[c]));
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
            H2V_TRY(h2v_domain_transform_dev(pk->dom, C2E, g.col(COEFF, 0, 1, pk->lookup_table[l0_]), n, scr, ne, 1));
            table_in_slot = pk->lookup_table[l0_];
        }
        uint32_t l1_ = l0_;
        src.clear();
        while (l1_ < L && pk->lookup_table[l1_] == table_in_slot && src.size() + 1 < SC) src.push_back(g.col(COEFF, 0, 0, pk->lookup_input[l1_++]));
        H2V_TRY(extend(src, scr + ne));
        mark(t_ext);
        for (uint32_t l = l0_; l < l1_; ++l)
            H2V_TRY(h2v_quotient_lookup_dev(pk->dom, h_ext, u64(y), u64(beta), u64(gamma), scr + (size_t)(1 + l - l0_) * ne, scr,
                                            pk->pa_E.as<fe>() + (size_t)l * ne, pk->ps_E.as<fe>() + (size_t)l * ne, pk->zl_E.as<fe>() + (size_t)l * ne, l0, ll, la));
        mark(t_fold);
        l0_ = l1_;
    }
    if (timing) fprintf(stderr, "evaluate_h (streamed): coeff_to_extended of the slices %.1f ms, folds %.1f ms\n", t_ext, t_fold);
    return H2V_OK;
}

//      steps 9-11: h_ext of proof p at hq + p ne, zeroed, then evaluate_h; its quotient after the division at hq + (B + p) ne
int evaluate_h(Group &g) {
    h2v_pk *pk = g.pk;
    H2V_TRY(pk->hq.ensure(2 * g.B * g.ne * sizeof(fe)));
    fe *h_ext = pk->hq.as<fe>(), *h_out = h_ext + g.B * g.ne;
    H2V_CU(cudaMemsetAsync(h_ext, 0, g.B * g.ne * sizeof(fe), pk->st));
    H2V_TRY(sync(pk));
    return pk->stream_ext ? evaluate_h_streamed(g, h_ext, h_out) : evaluate_h_resident(g, h_ext);
}

//      vanishing/prover.rs Committed::construct: h divided by the vanishing polynomial (back in coefficients), one blind
//      per piece, the NH pieces of n coefficients committed and written
int commit_quotient(Group &g) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, ne = g.ne, NH = g.NH;
    fe *h_ext = pk->hq.as<fe>(), *h_out = h_ext + B * ne;
    H2V_TRY(h2v_domain_transform_dev(pk->dom, H2V_OP_DIVIDE_BY_VANISHING, h_ext, ne, h_out, ne, B));
    for (auto &s : g.P)
        for (size_t i = 0; i < NH; ++i) (void)s->rng.fr_random();     // h_blinds
    // the B x NH pieces as contiguous columns of n (they already are when NH n = ne, and for one proof)
    g.pieces = h_out;
    if (B > 1 && NH * n != ne) {
        H2V_TRY(pk->hx_pieces.ensure(B * NH * n * sizeof(fe)));
        g.pieces = pk->hx_pieces.as<fe>();
        H2V_CU(cudaMemcpy2DAsync(g.pieces, NH * n * sizeof(fe), h_out, ne * sizeof(fe), NH * n * sizeof(fe), B, cudaMemcpyDeviceToDevice, pk->st));
        H2V_TRY(sync(pk));
    }
    H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, g.pieces, B * NH, g.pts));
    return write_commitments(g, g.pts, NH, false);
}

// ---- phase 5.  plonk/prover.rs create_proof step 12: x, h(X) = sum_i xn^i h_i(X) (vanishing/prover.rs
//      Constructed::evaluate), and every (polynomial, point) pair that is evaluated.  The list is the same for every
//      proof, over its own columns: in transcript order first, then the two the transcript skips.
struct Evaluations {
    std::vector<EvalPair> pairs;     // NE per proof; .point indexes the proof's NPT distinct points x w^rot
    std::vector<Fr64> evals;         // of the pairs
    std::vector<Fr64> points;        // proof p's at p NPT
    size_t NE = 0, NPT = 0;
    std::vector<uint32_t> queries;   // the pairs (of one proof) in the order upstream's prover queries them
};
int evaluations(Group &g, Evaluations &ev) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n;
    const uint32_t L = g.L, NP = g.NP, NS = g.NS;
    for (auto &s : g.P) {
        s->x = s->T.squeeze_challenge();
        s->xn = s->x;
        for (uint32_t i = 0; i < pk->k; ++i) s->xn = frh::sqr(s->xn);
    }
    // distinct evaluation points x * w^rot: the same rotations for every proof, in order of first use
    std::vector<int32_t> rots;
    auto point_of = [&](int32_t rot) -> uint32_t {
        for (size_t i = 0; i < rots.size(); ++i)
            if (rots[i] == rot) return (uint32_t)i;
        rots.push_back(rot);
        return (uint32_t)(rots.size() - 1);
    };
    const uint32_t p_cur = point_of(0), p_next = point_of(1), p_prev = point_of(-1), p_last = point_of(-(int32_t)(g.bf + 1));
    // h(X) of proof p at sh_h + p n
    H2V_TRY(pk->sh_h.ensure(2 * B * n * sizeof(fe)));
    fe *h_poly0 = pk->sh_h.as<fe>();
    H2V_TRY(sum_powers(g, g.pieces, g.NH, &ProofState::xn, h_poly0));
    std::vector<EvalPair> &pairs = ev.pairs;
    uint32_t e_random = 0, e_perm = 0, e_lookup = 0, n_written = 0, e_h = 0;
    for (size_t p = 0; p < B; ++p) {
        const size_t base = pairs.size();
        auto push = [&](const fe *poly, uint32_t pt) { pairs.push_back(EvalPair{poly, pt}); return (uint32_t)(pairs.size() - 1 - base); };
        const fe *z_C = pk->z_C.as<fe>() + p * NS * n, *zl_C = pk->zl_C.as<fe>() + p * L * n, *pa_C = pk->pa_C.as<fe>() + p * L * n,
                 *ps_C = pk->ps_C.as<fe>() + p * L * n;
        for (size_t q = 0; q < pk->aq_col.size(); ++q) push(g.col(COEFF, p, 0, pk->aq_col[q]), point_of(pk->aq_rot[q]));
        for (size_t q = 0; q < pk->fq_col.size(); ++q) push(g.col(COEFF, p, 1, pk->fq_col[q]), point_of(pk->fq_rot[q]));
        e_random = push(pk->rnd_C.as<fe>() + p * n, p_cur);
        for (uint32_t c = 0; c < NP; ++c) push(pk->sigma_C.as<fe>() + (size_t)c * n, p_cur);
        e_perm = e_random + 1 + NP;
        for (uint32_t s = 0; s < NS; ++s) {
            push(z_C + (size_t)s * n, p_cur);
            push(z_C + (size_t)s * n, p_next);
            if (s + 1 < NS) push(z_C + (size_t)s * n, p_last);
        }
        e_lookup = e_perm + (NS ? 3 * NS - 1 : 0);
        for (uint32_t l = 0; l < L; ++l) {
            push(zl_C + (size_t)l * n, p_cur);
            push(zl_C + (size_t)l * n, p_next);
            push(pa_C + (size_t)l * n, p_cur);
            push(pa_C + (size_t)l * n, p_prev);
            push(ps_C + (size_t)l * n, p_cur);
        }
        n_written = e_lookup + 5 * L;
        e_h = push(h_poly0 + p * n, p_cur);       // h(x): opened by the multi-open argument, not written
    }
    ev.NE = e_h + 1;
    ev.NPT = rots.size();
    // the queries of the multi-open argument in upstream's order: advice; permutation products
    // (permutation::prover::Evaluated::open: (x, z_s), (wx, z_s) for every set, then (w^last x, z_s) for all but the last
    // set taken in reverse order); lookups (lookup::prover::Evaluated::open: (x, z), (x, a'), (x, s'), (w^-1 x, a'),
    // (wx, z)); fixed; sigma; vanishing (h, then the random polynomial)
    std::vector<uint32_t> &q = ev.queries;
    for (uint32_t e = 0; e < pk->aq_col.size(); ++e) q.push_back(e);
    for (uint32_t s = 0; s < NS; ++s) q.insert(q.end(), {e_perm + 3 * s, e_perm + 3 * s + 1});
    for (uint32_t s = NS; s-- > 0;)
        if (s + 1 < NS) q.push_back(e_perm + 3 * s + 2);
    for (uint32_t l = 0; l < L; ++l) {
        const uint32_t b = e_lookup + 5 * l;
        q.insert(q.end(), {b, b + 2, b + 4, b + 3, b + 1});
    }
    for (uint32_t e = 0; e < pk->fq_col.size(); ++e) q.push_back((uint32_t)pk->aq_col.size() + e);
    for (uint32_t c = 0; c < NP; ++c) q.push_back(e_random + 1 + c);
    q.insert(q.end(), {e_h, e_random});
    const size_t NE = ev.NE, NPT = ev.NPT;
    ev.points.resize(B * NPT);
    for (size_t p = 0; p < B; ++p)
        for (size_t i = 0; i < NPT; ++i) ev.points[p * NPT + i] = frh::rotate(g.P[p]->x, pk->omega, pk->omega_inv, rots[i]);
    std::vector<EvalPair> dev_pairs(pairs);
    for (size_t e = 0; e < dev_pairs.size(); ++e) dev_pairs[e].point += (uint32_t)((e / NE) * NPT);
    ev.evals.resize(pairs.size());
    H2V_TRY(put(pk, pk->pairs, dev_pairs));
    H2V_TRY(put(pk, pk->pts, ev.points));
    H2V_TRY(pk->evals.ensure(pairs.size() * sizeof(fe)));
    eval_pairs_kernel<<<(unsigned)pairs.size(), 256, 0, pk->st>>>((const EvalPair *)pk->pairs.p, pk->pts.as<fe>(), (uint32_t)n, pk->evals.as<fe>());
    H2V_LAUNCHED();
    H2V_CU(cudaMemcpyAsync(ev.evals.data(), pk->evals.p, pairs.size() * sizeof(fe), cudaMemcpyDeviceToHost, pk->st));
    H2V_TRY(sync(pk));
    for (size_t p = 0; p < B; ++p)
        for (uint32_t i = 0; i < n_written; ++i) g.P[p]->T.write_scalar(ev.evals[p * NE + i]);
    return H2V_OK;
}

// ---- phase 6.  The multi-open argument, poly/kzg/multiopen/shplonk/prover.rs ProverSHPLONK::create_proof.  Every proof
//      has the same rotation sets (commitments grouped by the rotations they are opened at, in order of first
//      appearance); only the numeric order of the points inside a set differs.
struct RSet { uint64_t mask; std::vector<const fe *> polys; };
struct MultiOpen {
    std::vector<RSet> rsets;
    std::vector<Fr64> sorted_pts;
    uint64_t super_mask = 0;
    std::vector<std::vector<Fr64>> r_comb;                 // sum_j y^j R_ij(X), low degree
    std::vector<std::vector<std::vector<Fr64>>> r_ij;
    std::vector<std::vector<Fr64>> set_pts;                // the points of set i, numeric order
    std::vector<std::vector<Fr64>> ypow;
    std::vector<Fr64> pts_of(uint64_t mask) const {
        std::vector<Fr64> v;
        for (size_t r = 0; r < sorted_pts.size(); ++r)
            if ((mask >> r) & 1) v.push_back(sorted_pts[r]);
        return v;
    }
};

//      The host side for proof p (one host thread per proof): shplonk.rs construct_intermediate_sets, y / v, the Lagrange
//      bases and the interpolated R_ij
MultiOpen multi_open_sets(Group &g, const Evaluations &ev, size_t p) {
    const size_t NPT = ev.NPT;
    MultiOpen mo;
    const EvalPair *pr = ev.pairs.data() + p * ev.NE;
    const Fr64 *val = ev.evals.data() + p * ev.NE, *pt = ev.points.data() + p * NPT;
    // construct_intermediate_sets: point sets are ordered sets of field elements (BTreeSet<Fr>: numeric order of the
    // canonical values); commitments and rotation sets keep their order of first appearance
    std::vector<uint32_t> rank(NPT), ord(NPT);      // rank[i] = position of point i in the numeric order
    for (size_t i = 0; i < NPT; ++i) ord[i] = (uint32_t)i;
    std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return frh::less_canonical(pt[a], pt[b]); });
    for (size_t i = 0; i < NPT; ++i) rank[ord[i]] = (uint32_t)i;
    // a polynomial is identified by its device address, as upstream's PolynomialPointer
    struct Com { const fe *poly; uint64_t mask; };       // mask over ranks
    std::vector<Com> coms;
    std::map<const fe *, size_t> com_of;
    std::map<std::pair<const fe *, uint32_t>, Fr64> eval_of;
    for (uint32_t e : ev.queries) {
        const uint64_t bit = (uint64_t)1 << rank[pr[e].point];
        mo.super_mask |= bit;
        auto it = com_of.find(pr[e].poly);
        if (it == com_of.end()) {
            com_of[pr[e].poly] = coms.size();
            coms.push_back(Com{pr[e].poly, bit});
        } else {
            coms[it->second].mask |= bit;
        }
        eval_of[{pr[e].poly, rank[pr[e].point]}] = val[e];
    }
    for (const Com &c : coms) {
        size_t i = 0;
        for (; i < mo.rsets.size(); ++i)
            if (mo.rsets[i].mask == c.mask) break;
        if (i == mo.rsets.size()) mo.rsets.push_back(RSet{c.mask, {}});
        mo.rsets[i].polys.push_back(c.poly);
    }
    mo.sorted_pts.resize(NPT);
    for (size_t i = 0; i < NPT; ++i) mo.sorted_pts[rank[i]] = pt[i];
    ProofState &S = *g.P[p];
    S.ys = S.T.squeeze_challenge();
    S.vs = S.T.squeeze_challenge();
    const size_t NR = mo.rsets.size();
    mo.r_comb.resize(NR);
    mo.r_ij.resize(NR);
    mo.set_pts.resize(NR);
    mo.ypow.resize(NR);
    for (size_t i = 0; i < NR; ++i) {
        const std::vector<Fr64> ps = mo.pts_of(mo.rsets[i].mask);
        const size_t m = ps.size(), nc = mo.rsets[i].polys.size();
        const std::vector<std::vector<Fr64>> basis = lagrange_basis(ps);
        Fr64 cur = frh::ONE;
        mo.r_comb[i].assign(m, frh::zero());
        mo.r_ij[i].resize(nc);
        mo.ypow[i].resize(nc);
        for (size_t j = 0; j < nc; ++j) {
            mo.ypow[i][j] = cur;
            std::vector<Fr64> evj;
            for (size_t r = 0; r < NPT; ++r)
                if ((mo.rsets[i].mask >> r) & 1) evj.push_back(eval_of[{mo.rsets[i].polys[j], (uint32_t)r}]);
            mo.r_ij[i][j] = lagrange_interpolate(basis, evj);
            for (size_t t = 0; t < m; ++t) mo.r_comb[i][t] = frh::add(mo.r_comb[i][t], frh::mul(mo.r_ij[i][j][t], cur));
            cur = frh::mul(cur, S.ys);
        }
        mo.set_pts[i] = ps;
    }
    return mo;
}

//      The device side for the group: S_i = sum_j y^j P_ij, Q_i = (S_i - sum_j y^j R_ij) / prod (X - p), h = sum_i v^i Q_i
//      (committed), u, then L(X) and W = L / (X - u) / z_0 (committed)
int shplonk(Group &g, const std::vector<MultiOpen> &MO) {
    h2v_pk *pk = g.pk;
    const size_t B = g.B, n = g.n, NR = MO[0].rsets.size();
    for (const MultiOpen &mo : MO)
        if (mo.rsets.size() != NR) return failf(H2V_EINVAL, "create_proof: rotation sets differ between the proofs of a group");
    size_t max_m = 1;
    for (size_t i = 0; i < NR; ++i) max_m = std::max(max_m, MO[0].set_pts[i].size());
    H2V_TRY(pk->sh_S.ensure(B * NR * n * sizeof(fe)));
    H2V_TRY(pk->sh_A.ensure((B * n + 8) * sizeof(fe)));
    H2V_TRY(pk->sh_B.ensure(std::max<size_t>(B * NR, B) * n * sizeof(fe)));
    fe *S0 = pk->sh_S.as<fe>(), *Q = pk->sh_B.as<fe>();       // S_i and the quotient contributions Q_i of proof p: (p NR + i) n
    fe *hx0 = pk->sh_h.as<fe>() + B * n;                      // proof p's h(X) at hx0 + p n
    {
        // S_i(X) = sum_j y^j P_ij(X) for every proof and set in one launch; N_i = S_i - sum_j y^j R_ij
        std::vector<const fe *> hp;
        std::vector<Fr64> cf, low(B * NR * max_m, frh::zero());
        std::vector<uint32_t> off;
        for (size_t p = 0; p < B; ++p)
            for (size_t i = 0; i < NR; ++i) {
                off.push_back((uint32_t)hp.size());
                hp.insert(hp.end(), MO[p].rsets[i].polys.begin(), MO[p].rsets[i].polys.end());
                cf.insert(cf.end(), MO[p].ypow[i].begin(), MO[p].ypow[i].end());
                std::copy(MO[p].r_comb[i].begin(), MO[p].r_comb[i].end(), low.begin() + (p * NR + i) * max_m);
            }
        off.push_back((uint32_t)hp.size());
        H2V_TRY(lincomb(pk, hp, cf, off, S0, n, n));
        H2V_CU(cudaMemcpyAsync(Q, S0, B * NR * n * sizeof(fe), cudaMemcpyDeviceToDevice, pk->st));
        H2V_TRY(sub_low(pk, Q, n, low, B * NR));
        H2V_TRY(sync(pk));
    }
    // Q_i = N_i / prod (X - p): one division per point of the set, every (proof, set) with a t-th point in one batched
    // pass; each column ping-pongs between its home in Q and its own slot in sh_T
    H2V_TRY(pk->sh_T.ensure(B * NR * n * sizeof(fe)));
    std::vector<KateJob> jobs;
    for (size_t t = 0; t < max_m; ++t) {
        jobs.clear();
        for (size_t p = 0; p < B; ++p)
            for (size_t i = 0; i < NR; ++i) {
                const std::vector<Fr64> &ps = MO[p].set_pts[i];
                if (t >= ps.size()) continue;
                fe *home = Q + (p * NR + i) * n, *slot = pk->sh_T.as<fe>() + (p * NR + i) * n;
                KateJob j{t % 2 ? slot : home, t % 2 ? home : slot, n - t, {}};
                memcpy(j.b, u64(ps[t]), sizeof j.b);
                jobs.push_back(j);
            }
        H2V_TRY(kate_division_batch_dev(jobs.data(), jobs.size()));
    }
    for (size_t p = 0; p < B; ++p)
        for (size_t i = 0; i < NR; ++i) {
            const size_t m = MO[p].set_pts[i].size(), len = n - m;
            fe *home = Q + (p * NR + i) * n;
            if (m % 2) H2V_CU(cudaMemcpyAsync(home, pk->sh_T.as<fe>() + (p * NR + i) * n, len * sizeof(fe), cudaMemcpyDeviceToDevice, pk->st));
            H2V_CU(cudaMemsetAsync(home + len, 0, m * sizeof(fe), pk->st));
        }
    H2V_TRY(sum_powers(g, Q, NR, &ProofState::vs, hx0));      // h(X) = sum_i v^i Q_i(X)
    H2V_TRY(sync(pk));
    H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, hx0, B, g.pts));
    H2V_TRY(write_commitments(g, g.pts, 1, false));
    for (auto &s : g.P) s->uc = s->T.squeeze_challenge();
    // L(X) = sum_i v^i z_i (S_i(X) - sum_j y^j R_ij(u)) - Z_T(u) h(X);  second opening proof = L / (X - u) / z_0
    std::vector<const fe *> hp(B * (NR + 1));
    std::vector<Fr64> cf(B * (NR + 1)), konst(B), z0inv(B);
    std::vector<uint32_t> off(B + 1);
    H2V_TRY(par_proofs(B, [&](size_t p) -> int {
        const MultiOpen &mo = MO[p];
        const Fr64 &uc = g.P[p]->uc;
        Fr64 vp = frh::ONE, z0 = frh::ONE;
        konst[p] = frh::zero();
        for (size_t i = 0; i < NR; ++i) {
            Fr64 zi = frh::ONE;
            for (size_t r = 0; r < mo.sorted_pts.size(); ++r)
                if (((mo.super_mask & ~mo.rsets[i].mask) >> r) & 1) zi = frh::mul(zi, frh::sub(uc, mo.sorted_pts[r]));
            if (i == 0) z0 = zi;
            Fr64 ri = frh::zero(), yp = frh::ONE;
            for (size_t j = 0; j < mo.rsets[i].polys.size(); ++j) {
                ri = frh::add(ri, frh::mul(yp, eval_small(mo.r_ij[i][j], uc)));
                yp = frh::mul(yp, g.P[p]->ys);
            }
            hp[p * (NR + 1) + i] = S0 + (p * NR + i) * n;
            cf[p * (NR + 1) + i] = frh::mul(vp, zi);
            konst[p] = frh::add(konst[p], frh::mul(cf[p * (NR + 1) + i], ri));
            vp = frh::mul(vp, g.P[p]->vs);
        }
        Fr64 zt = frh::ONE;
        for (const Fr64 &x : mo.pts_of(mo.super_mask)) zt = frh::mul(zt, frh::sub(uc, x));
        hp[p * (NR + 1) + NR] = hx0 + p * n;
        cf[p * (NR + 1) + NR] = frh::neg(zt);
        off[p] = (uint32_t)(p * (NR + 1));
        z0inv[p] = frh::inv(z0);
        return H2V_OK;
    }));
    off[B] = (uint32_t)(B * (NR + 1));
    fe *Lx = pk->sh_A.as<fe>();           // proof p's L at Lx + p n
    H2V_TRY(lincomb(pk, hp, cf, off, Lx, n, n));
    H2V_TRY(sub_low(pk, Lx, n, konst, B));
    H2V_TRY(sync(pk));
    fe *W = Q;        // the quotient contributions are no longer needed; proof p's W at W + p n
    jobs.resize(B);
    for (size_t p = 0; p < B; ++p) {
        jobs[p] = KateJob{Lx + p * n, W + p * n, n, {}};
        memcpy(jobs[p].b, u64(g.P[p]->uc), sizeof jobs[p].b);
    }
    H2V_TRY(kate_division_batch_dev(jobs.data(), B));
    for (size_t p = 0; p < B; ++p) H2V_CU(cudaMemsetAsync(W + p * n + (n - 1), 0, sizeof(fe), pk->st));
    H2V_TRY(put(pk, pk->scal, z0inv));
    scale_cols_kernel<<<dim3(g.gn, (unsigned)B), 256, 0, pk->st>>>(W, (uint32_t)n, pk->scal.as<fe>());
    H2V_LAUNCHED();
    H2V_TRY(sync(pk));
    H2V_TRY(commit_dev(pk, H2V_BASIS_MONOMIAL, W, B, g.pts));
    return write_commitments(g, g.pts, 1, false);
}

// The prover: a group of B proofs phase by phase, each phase ended by lap() (h2v_pk_last_phase_ms).  The caller holds
// pk->mu and has checked the inputs; on a failure traced to one proof, `bad` is that proof (else it stays SIZE_MAX).
int prove_group(h2v_pk *pk, size_t B, const ProofIn *in, const Generated *gen, std::vector<std::vector<uint8_t>> &proofs, size_t &bad) {
    Group g(pk, B, in, gen, bad);
    H2V_TRY(instances_and_advice(g));
    g.lap();   // phase 0: upload (or generation) + advice commitments
    H2V_TRY(permuted_lookups(g));
    g.lap();   // phase 1: lookup permutations
    H2V_TRY(permutation_products(g));
    H2V_TRY(lookup_products(g));
    g.lap();   // phase 2: grand products
    H2V_TRY(random_polynomial(g));
    H2V_TRY(transform_columns(g));
    for (auto &s : g.P) s->y = s->T.squeeze_challenge();
    g.lap();   // phase 3: random poly + transforms
    H2V_TRY(evaluate_h(g));
    H2V_TRY(commit_quotient(g));
    g.lap();   // phase 4: evaluate_h + quotient commitments
    Evaluations ev;
    H2V_TRY(evaluations(g, ev));
    g.lap();   // phase 5: evaluations
    std::vector<MultiOpen> mo(B);
    H2V_TRY(par_proofs(B, [&](size_t p) -> int {
        mo[p] = multi_open_sets(g, ev, p);
        return H2V_OK;
    }));
    H2V_TRY(shplonk(g, mo));
    g.lap();   // phase 6: multi-open argument
    proofs.resize(B);
    for (size_t p = 0; p < B; ++p) proofs[p].swap(g.P[p]->T.out);
    return H2V_OK;
}

// ---------------------------------------------------------------- groups
// device bytes one proof of a group adds (the rotation sets of the multi-open argument are counted as 8)
size_t proof_bytes(const h2v_pk *pk) {
    const size_t n = pk->n, ne = pk->ne, L = pk->lookup_input.size(), NS = pk->n_sets;
    const size_t cols = pk->n_advice + pk->n_instance + 3 * L + NS;              // Lagrange, coefficient and extended forms
    const size_t ncols = 2 * std::max(NS, L) + 1 + (pk->degree - 1) + 2 + 2 * 8 + 1;   // num / den, random, pieces, h, S / Q, L
    return sizeof(fe) * (cols * (2 * n + (pk->stream_ext ? 0 : ne)) + 2 * ne + ncols * n) + 4096;
}
// The group size for n_items items (proofs, or witnesses to check) of item_bytes device bytes each: H2V_PROOF_GROUP if
// set, else as many as fit in the device memory left after the key, with 8 GB kept free as the extended-sigma cache
// keeps it; at most `cap`, the largest group every grid dimension and batch call allows.  extra_held: device bytes
// outside the key's workspace that the groups reuse.
size_t group_size(h2v_pk *pk, size_t n_items, size_t item_bytes, size_t cap, size_t extra_held = 0) {
    size_t held = extra_held;
    for (size_t i = 0; DevBuf *b = workspace(pk, i); ++i) held += b->cap;
    return group_size_free(n_items, item_bytes, cap, held);
}
// ... for n_proofs proofs, each also needing extra_bytes (a witness program's evaluation).  Streamed keys prove one at a time.
size_t proof_group_size(h2v_pk *pk, size_t n_proofs, size_t extra_bytes = 0, size_t extra_held = 0) {
    if (pk->stream_ext || n_proofs <= 1) return 1;
    const size_t cmax = std::max<size_t>({pk->n_sets, pk->lookup_input.size(), 16});
    return group_size(pk, n_proofs, proof_bytes(pk) + extra_bytes, std::min<size_t>(65535 / cmax, (((size_t)1 << 31) - 1) / (pk->n * cmax)),
                      extra_held);
}

// Inputs of proof `idx` (who: the prefix of the error text)
int check_inputs(const h2v_pk *pk, const ProofIn &in, const std::string &who) {
    if (!in.seed) return failf(H2V_EINVAL, "%s: NULL rng seed", who.c_str());
    if ((pk->n_advice && !in.advice) || (pk->n_instance && (!in.instances || !in.instance_len)))
        return failf(H2V_EINVAL, "%s: NULL column list", who.c_str());
    for (uint32_t c = 0; c < pk->n_advice; ++c)
        if (!in.advice[c]) return failf(H2V_EINVAL, "%s: advice[%u] is NULL", who.c_str(), c);
    for (uint32_t c = 0; c < pk->n_instance; ++c) {
        if (in.instance_len[c] > pk->u)
            return failf(H2V_EINVAL, "%s: InstanceTooLarge (%u values, %u usable rows)", who.c_str(), in.instance_len[c], pk->u);
        if (in.instance_len[c] && !in.instances[c]) return failf(H2V_EINVAL, "%s: instances[%u] is NULL", who.c_str(), c);
    }
    return H2V_OK;
}

// The key's opportunistic cache of extended sigma columns (streamed mode) took memory something else now needs: give it
// back for good, if it holds any, so that the caller runs its step again
bool release_sigma_cache(h2v_pk *pk) {
    if (!pk->cached_sigma) return false;
    cudaStreamSynchronize(pk->st);
    pk->ext_cache.release();
    pk->cached_sigma = 0;
    return true;
}

// n_proofs proofs in groups; emit(i, bytes) receives proof i.  A group that runs out of device memory is halved and run
// again (a group of one needs what one proof always needed).  `who` (NULL for h2v_create_proof): prefix error texts
// with the call and the proof they concern.  gen: the columns come from a witness program, bound to the key's device
// here, under its mutex (taken after the key's).
template <class Emit> int run_proofs(h2v_pk *pk, size_t n_proofs, const ProofIn *in, const char *who, const Generated *gen, Emit emit) {
    H2V_TRY(set_device(pk->dev, who ? who : "create_proof"));
    std::lock_guard<std::mutex> lk(pk->mu);
    std::unique_lock<std::mutex> lk_prog;
    size_t gen_bytes = 0, gen_held = 0;
    if (gen) {
        lk_prog = std::unique_lock<std::mutex>(witness_program_mutex(gen->prog));
        H2V_TRY(witness_program_bind(gen->prog, pk->dev, pk->st, who, &gen_held));
        gen_bytes = witness_eval_bytes(gen->prog);
    }
    for (double &v : pk->last_ms) v = 0;
    size_t G = proof_group_size(pk, n_proofs, gen_bytes, gen_held);
    for (size_t p0 = 0; p0 < n_proofs;) {
        const size_t b = std::min(G, n_proofs - p0);
        std::vector<std::vector<uint8_t>> out;
        size_t bad = SIZE_MAX;
        const Generated gen_b = gen ? gen->at(p0) : Generated{};
        int rc = prove_group(pk, b, in + p0, gen ? &gen_b : nullptr, out, bad);
        if (rc == H2V_ENOMEM && release_sigma_cache(pk)) continue;
        if (rc == H2V_ENOMEM && b > 1) {
            cudaStreamSynchronize(pk->st);
            for (size_t i = 0; DevBuf *w = workspace(pk, i); ++i) w->release();
            G = b / 2;
            continue;
        }
        if (rc) {
            cudaStreamSynchronize(pk->st);
            if (who) {
                const std::string msg = h2v_last_error();
                if (bad != SIZE_MAX) return failf(rc, "%s: %s %zu: %s", who, gen ? "witness" : "proof", p0 + bad, msg.c_str());
                return failf(rc, "%s: group of proofs %zu .. %zu: %s", who, p0, p0 + b - 1, msg.c_str());
            }
            return rc;
        }
        for (size_t p = 0; p < b; ++p) H2V_TRY(emit(p0 + p, out[p]));
        pk->last_ms[7] += 1;      // groups run
        p0 += b;
    }
    return H2V_OK;
}

// the key's constraint system, as h2v_pk_load received it
h2v_circuit_t circuit_of(const h2v_pk *pk) {
    h2v_circuit_t cs{};
    cs.k = pk->k;
    cs.degree = pk->degree;
    cs.blinding_factors = pk->bf;
    cs.n_advice = pk->n_advice;
    cs.n_fixed = pk->n_fixed;
    cs.n_instance = pk->n_instance;
    cs.n_gates = (uint32_t)pk->gate_advice.size();
    cs.gate_advice = pk->gate_advice.data();
    cs.gate_selector = pk->gate_selector.data();
    cs.n_lookups = (uint32_t)pk->lookup_input.size();
    cs.lookup_input = pk->lookup_input.data();
    cs.lookup_table = pk->lookup_table.data();
    cs.n_perm = (uint32_t)pk->perm_kind.size();
    cs.perm_kind = pk->perm_kind.data();
    cs.perm_index = pk->perm_index.data();
    cs.n_advice_queries = (uint32_t)pk->aq_col.size();
    cs.advice_query_col = pk->aq_col.data();
    cs.advice_query_rot = pk->aq_rot.data();
    cs.n_fixed_queries = (uint32_t)pk->fq_col.size();
    cs.fixed_query_col = pk->fq_col.data();
    cs.fixed_query_rot = pk->fq_rot.data();
    return cs;
}

// run_proofs' emit for proofs written to out + p stride
auto proofs_to(uint8_t *out, size_t stride, size_t size, const char *who) {
    return [=](size_t p, const std::vector<uint8_t> &proof) -> int {
        if (proof.size() != size) return failf(H2V_EINVAL, "%s: proof %zu has %zu bytes, expected %zu", who, p, proof.size(), size);
        memcpy(out + p * stride, proof.data(), size);
        return H2V_OK;
    };
}

// n_witnesses witnesses checked in groups against the key's tables, as run_proofs runs proofs: stage(w0, b, ms, bad)
// puts witnesses w0 .. w0 + b - 1 into adv_L / inst_L (ms[0] += its time; bad: the witness of the group a failure is
// traced to).  Each witness also needs extra_bytes of device memory, and extra_held bytes outside the key's workspace
// are reused by the groups.  The caller holds pk->mu and has checked the arguments.
template <class Stage>
int run_mock(h2v_pk *pk, size_t n_witnesses, const char *who, size_t extra_bytes, size_t extra_held, h2v_mock_failure_t *failures_out,
             size_t cap, uint64_t *n_failures, Stage stage) {
    const h2v_circuit_t cs = circuit_of(pk);
    double ms[2] = {0, 0};
    while (!pk->mock) {      // the key tables, on the first call
        const double t = now_ms();
        const int rc = mock_key_build(pk->st, &cs, pk->fixed_L.as<fe>(), pk->sigma_L.as<fe>(), &pk->mock);
        ms[1] += now_ms() - t;
        if (rc == H2V_ENOMEM && release_sigma_cache(pk)) continue;
        if (rc) {
            cudaStreamSynchronize(pk->st);
            return rc;
        }
    }
    // the witnesses in groups, as run_proofs runs proofs; they are staged in the key's adv_L / inst_L workspace
    size_t G = group_size(pk, n_witnesses, mock_witness_bytes(*pk->mock) + extra_bytes, mock_max_batch(*pk->mock), extra_held);
    for (size_t w0 = 0; w0 < n_witnesses;) {
        const size_t b = std::min(G, n_witnesses - w0);
        size_t bad = SIZE_MAX;
        int rc = stage(w0, b, ms, bad);
        if (!rc)
            rc = mock_check(pk->st, *pk->mock, b, pk->adv_L.as<fe>(), pk->inst_L.as<fe>(), cap ? failures_out + w0 * cap : nullptr, cap,
                            n_failures + w0, ms);
        if (rc == H2V_ENOMEM && release_sigma_cache(pk)) continue;
        if (rc == H2V_ENOMEM && b > 1) {
            cudaStreamSynchronize(pk->st);
            for (size_t i = 0; DevBuf *w = workspace(pk, i); ++i) w->release();
            G = b / 2;
            continue;
        }
        if (rc) {
            cudaStreamSynchronize(pk->st);
            const std::string msg = h2v_last_error();
            if (bad != SIZE_MAX) return failf(rc, "%s: witness %zu: %s", who, w0 + bad, msg.c_str());
            return failf(rc, "%s: witnesses %zu .. %zu: %s", who, w0, w0 + b - 1, msg.c_str());
        }
        w0 += b;
    }
    mock_set_last_ms(ms);
    return H2V_OK;
}

// The argument checks of the _from_inputs calls that concern the program, in the order h2v.h states them; info: the
// program's h2v_witness_program_info
int check_program(const h2v_pk *pk, h2v_witness_program_t prog, size_t n_witnesses, size_t n_inputs, const uint64_t *inputs, const char *who,
                  uint64_t info[8]) {
    H2V_TRY(h2v_witness_program_info(prog, info));
    if (n_inputs != info[0])
        return failf(H2V_EINVAL, "%s: %zu inputs per witness, the program has %llu", who, n_inputs, (unsigned long long)info[0]);
    for (size_t w = 0; w < n_witnesses; ++w)
        for (size_t i = 0; i < n_inputs; ++i)
            if (!fr_reduced(inputs + 4 * (w * n_inputs + i)))
                return failf(H2V_EINVAL, "%s: witness %zu: input %zu is not a reduced Montgomery value", who, w, i);
    if (info[6] != pk->k) return failf(H2V_EINVAL, "%s: the program has k = %llu, the key k = %u", who, (unsigned long long)info[6], pk->k);
    if (info[4] != pk->n_advice)
        return failf(H2V_EINVAL, "%s: the program has %llu advice columns, the key %u", who, (unsigned long long)info[4], pk->n_advice);
    if (pk->n_instance > 1 || (pk->n_instance == 1 && info[5] > pk->u) || (pk->n_instance == 0 && info[5]))
        return failf(H2V_EINVAL, "%s: the program's %llu instances do not fit the key's %u instance columns of %u usable rows", who,
                     (unsigned long long)info[5], pk->n_instance, pk->u);
    return H2V_OK;
}

}  // namespace

extern "C" {

int h2v_create_proof(h2v_pk_t pk, const uint64_t *const *advice, const uint64_t *const *instances, const uint32_t *instance_len,
                     const uint8_t rng_seed[32], uint8_t *proof_out, size_t proof_cap, size_t *proof_len) {
    if (!pk || !rng_seed || !proof_len) return failf(H2V_EINVAL, "create_proof: NULL argument");
    const ProofIn in{advice, instances, instance_len, rng_seed};
    H2V_TRY(check_inputs(pk, in, "create_proof"));
    return run_proofs(pk, 1, &in, nullptr, nullptr, [&](size_t, const std::vector<uint8_t> &proof) -> int {
        *proof_len = proof.size();
        if (proof.size() > proof_cap || !proof_out)
            return failf(H2V_EINVAL, "create_proof: proof needs %zu bytes, buffer has %zu", proof.size(), proof_cap);
        memcpy(proof_out, proof.data(), proof.size());
        return H2V_OK;
    });
}
int h2v_create_proofs(h2v_pk_t pk, size_t n_proofs, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
                      const uint32_t *const *instance_len, const uint8_t *rng_seeds, uint8_t *proofs_out, size_t proof_stride) {
    if (!pk) return failf(H2V_EINVAL, "create_proofs: NULL key");
    if (!n_proofs) return H2V_OK;
    if (!rng_seeds || !proofs_out || (pk->n_advice && !advice) || (pk->n_instance && (!instances || !instance_len)))
        return failf(H2V_EINVAL, "create_proofs: NULL argument");
    const size_t size = h2v_proof_size(pk);
    if (proof_stride < size) return failf(H2V_EINVAL, "create_proofs: proof_stride %zu is shorter than a proof (%zu bytes)", proof_stride, size);
    std::vector<ProofIn> in(n_proofs);
    for (size_t p = 0; p < n_proofs; ++p) {
        in[p] = ProofIn{pk->n_advice ? advice[p] : nullptr, pk->n_instance ? instances[p] : nullptr, pk->n_instance ? instance_len[p] : nullptr,
                        rng_seeds + 32 * p};
        char who[64];
        snprintf(who, sizeof who, "create_proofs: proof %zu", p);
        H2V_TRY(check_inputs(pk, in[p], who));
    }
    return run_proofs(pk, n_proofs, in.data(), "create_proofs", nullptr, proofs_to(proofs_out, proof_stride, size, "create_proofs"));
}
int h2v_create_proofs_from_inputs(h2v_pk_t pk, h2v_witness_program_t prog, size_t n_proofs, size_t n_inputs, const uint64_t *inputs,
                                  const uint8_t *rng_seeds, uint8_t *proofs_out, size_t proof_stride, uint64_t *instances_out) {
    const char *who = "create_proofs_from_inputs";
    if (!pk || !prog) return failf(H2V_EINVAL, "%s: NULL key or program", who);
    if (!n_proofs) return H2V_OK;
    if ((n_inputs && !inputs) || !rng_seeds || !proofs_out) return failf(H2V_EINVAL, "%s: NULL argument", who);
    uint64_t info[8];
    H2V_TRY(check_program(pk, prog, n_proofs, n_inputs, inputs, who, info));
    const size_t size = h2v_proof_size(pk);
    if (proof_stride < size) return failf(H2V_EINVAL, "%s: proof_stride %zu is shorter than a proof (%zu bytes)", who, proof_stride, size);
    // the instances come back to the host for the transcripts: into instances_out, or a buffer of the call
    const size_t n_inst = info[5];
    std::vector<uint64_t> inst_own(instances_out ? 0 : n_proofs * n_inst * 4);
    uint64_t *inst = instances_out ? instances_out : inst_own.data();
    const uint32_t inst_len = (uint32_t)n_inst;
    std::vector<const uint64_t *> inst_col(n_proofs);
    std::vector<ProofIn> in(n_proofs);
    for (size_t p = 0; p < n_proofs; ++p) {
        inst_col[p] = inst + p * n_inst * 4;
        in[p] = ProofIn{nullptr, pk->n_instance ? &inst_col[p] : nullptr, pk->n_instance ? &inst_len : nullptr, rng_seeds + 32 * p};
    }
    const Generated gen{prog, n_inputs, n_inst, inputs, inst};
    return run_proofs(pk, n_proofs, in.data(), who, &gen, proofs_to(proofs_out, proof_stride, size, who));
}
int h2v_pk_mock_prover(h2v_pk_t pk, size_t n_witnesses, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
                       const uint32_t *const *instance_len, h2v_mock_failure_t *failures_out, size_t cap, uint64_t *n_failures) {
    if (!pk) return failf(H2V_EINVAL, "pk_mock_prover: NULL key");
    if (!n_witnesses) return H2V_OK;
    if (!n_failures || (cap && !failures_out) || (pk->n_advice && !advice) || (pk->n_instance && (!instances || !instance_len)))
        return failf(H2V_EINVAL, "pk_mock_prover: NULL argument");
    const h2v_circuit_t cs = circuit_of(pk);
    for (size_t w = 0; w < n_witnesses; ++w) {
        char who[64];
        snprintf(who, sizeof who, "pk_mock_prover: witness %zu", w);
        if ((pk->n_advice && !advice[w]) || (pk->n_instance && (!instances[w] || !instance_len[w])))
            return failf(H2V_EINVAL, "%s: NULL column list", who);
        if (pk->n_advice) H2V_TRY(mock_check_advice(&cs, advice[w], who));
        if (pk->n_instance) H2V_TRY(mock_check_instances(&cs, instances[w], instance_len[w], who));
    }
    H2V_TRY(mock_check_limits(&cs, "pk_mock_prover"));
    H2V_TRY(set_device(pk->dev, "pk_mock_prover"));
    std::lock_guard<std::mutex> lk(pk->mu);
    return run_mock(pk, n_witnesses, "pk_mock_prover", 0, 0, failures_out, cap, n_failures, [&](size_t w0, size_t b, double ms[2], size_t &) {
        return mock_stage(pk->st, *pk->mock, b, advice ? advice + w0 : nullptr, instances ? instances + w0 : nullptr,
                          instance_len ? instance_len + w0 : nullptr, pk->adv_L, pk->inst_L, ms);
    });
}
int h2v_pk_mock_prover_from_inputs(h2v_pk_t pk, h2v_witness_program_t prog, size_t n_witnesses, size_t n_inputs, const uint64_t *inputs,
                                   h2v_mock_failure_t *failures_out, size_t cap, uint64_t *n_failures) {
    const char *who = "pk_mock_prover_from_inputs";
    if (!pk || !prog) return failf(H2V_EINVAL, "%s: NULL key or program", who);
    if (!n_witnesses) return H2V_OK;
    if ((n_inputs && !inputs) || !n_failures || (cap && !failures_out)) return failf(H2V_EINVAL, "%s: NULL argument", who);
    uint64_t info[8];
    H2V_TRY(check_program(pk, prog, n_witnesses, n_inputs, inputs, who, info));
    const h2v_circuit_t cs = circuit_of(pk);
    H2V_TRY(mock_check_limits(&cs, who));
    H2V_TRY(set_device(pk->dev, who));
    std::lock_guard<std::mutex> lk(pk->mu);
    std::lock_guard<std::mutex> lk_prog(witness_program_mutex(prog));      // after the key's
    size_t held = 0;
    H2V_TRY(witness_program_bind(prog, pk->dev, pk->st, who, &held));
    const size_t n = pk->n, A = pk->n_advice, I = pk->n_instance;
    return run_mock(pk, n_witnesses, who, witness_eval_bytes(prog), held, failures_out, cap, n_failures,
                    [&](size_t w0, size_t b, double ms[2], size_t &bad) -> int {
                        const double t = now_ms();
                        H2V_TRY(pk->adv_L.ensure(b * A * n * sizeof(fe)));
                        H2V_TRY(pk->inst_L.ensure(std::max<size_t>(1, b * I) * n * sizeof(fe)));
                        size_t bad_w = b;
                        const int rc = witness_generate_dev(prog, pk->st, b, inputs + w0 * n_inputs * 4, pk->adv_L.as<fe>(), pk->inst_L.as<fe>(),
                                                            I ? n : 0, nullptr, &bad_w);
                        ms[0] += now_ms() - t;
                        if (bad_w < b) bad = bad_w;
                        return rc;
                    });
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
