// quotient.cuh -- the per-row part of the quotient evaluation on the extended coset
// ("next" row 1 of SURVEY.md 8(f)).
//
// Replaces the three row loops of halo2-axiom plonk/evaluation.rs `Evaluator::evaluate_h` [UPSTREAM; reached
// from /root/reference/src/scaffold/mod.rs:296 through gen_snark_shplonk -> create_proof], for the constraint
// system halo2-base builds (FlexGateConfig / RangeConfig, [UPSTREAM] gates/flex_gate.rs, gates/range.rs):
//   * custom gates: one "vertical" gate per advice column,  q(X) * (a(X) + a(wX) a(w^2 X) - a(w^3 X))
//   * the permutation argument over `chunk_len = degree - 2` columns per grand product
//   * the lookup argument (one compressed input / table expression pair per lookup)
// Every term is folded into the running value as  h <- h * y + term, in upstream's order; the arithmetic is
// exact field arithmetic, so the result is bit-identical whatever the evaluation strategy.
//
// Layout: every polynomial is a device-resident column of 2^extended_k Fr values (Montgomery), the output of
// coeff_to_extended; rotation r at row i reads row (i + r * 2^(extended_k - k)) mod 2^extended_k
// (upstream `get_rotation_idx`).  One thread per row; a row costs 3 products per gate, 4 per permuted column and
// 13 per lookup, against 64-128 bytes of column reads per term: multiplier-bound like the NTT.
#pragma once
#include "ff.cuh"

namespace h2v {

typedef FrP FrQ;

struct QuotientCommon {
    uint32_t n_ext;     // 2^extended_k
    uint32_t rot;       // 2^(extended_k - k): rows per unit rotation
};

// A group of proofs on one key: proof p (grid.y) folds into h + p * h_stride with its own y, beta, gamma
// (scal[3p], scal[3p + 1], scal[3p + 2]); a public entry point is a group of one.
struct QuotientGroup {
    fe *h;
    size_t h_stride;
    const fe *scal;
};

__device__ __forceinline__ uint32_t q_rot(uint32_t idx, int r, const QuotientCommon &c) {
    return (idx + (uint32_t)(r * (int)c.rot)) & (c.n_ext - 1);
}

// a set of equally long device columns: either `stride` elements apart from a base, or through a device-resident
// table of column pointers (the prover's columns live in several allocations: advice, fixed, instance); proof p's set
// starts `pstride` elements / table entries after proof p-1's
struct ColsStrided {
    const fe *base;
    size_t stride, pstride;
    __device__ __forceinline__ const fe *col(uint32_t j) const { return base + (size_t)j * stride; }
    __device__ __forceinline__ ColsStrided at(uint32_t p) const { return ColsStrided{base + p * pstride, stride, 0}; }
};
struct ColsTable {
    const fe *const *ptrs;
    size_t pstride;
    __device__ __forceinline__ const fe *col(uint32_t j) const { return ptrs[j]; }
    __device__ __forceinline__ ColsTable at(uint32_t p) const { return ColsTable{ptrs + p * pstride, 0}; }
};

// h[i] = fold_j ( q_j[i] * (a_j[i] + a_j[i+r] * a_j[i+2r] - a_j[i+3r]) )
template <class QC, class AC>
__global__ void __launch_bounds__(256) quotient_gates_kernel(QuotientGroup g, QuotientCommon c, uint32_t n_gates, QC qs, AC as) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (idx >= c.n_ext) return;
    const QC q = qs.at(p);
    const AC a = as.at(p);
    fe *h = g.h + p * g.h_stride;
    const fe y = fe_load_global(g.scal + 3 * p);
    const uint32_t i1 = q_rot(idx, 1, c), i2 = q_rot(idx, 2, c), i3 = q_rot(idx, 3, c);
    fe v = fe_load_global(h + idx);
    for (uint32_t j = 0; j < n_gates; ++j) {
        const fe *aj = a.col(j);
        fe t = fe_mul<FrQ>(fe_load_global(aj + i1), fe_load_global(aj + i2));
        t = fe_sub<FrQ>(fe_add<FrQ>(fe_load_global(aj + idx), t), fe_load_global(aj + i3));
        t = fe_mul<FrQ>(t, fe_load_global(q.col(j) + idx));
        v = fe_add<FrQ>(fe_mul<FrQ>(v, y), t);
    }
    fe_store_global(h + idx, v);
}

struct QuotientPerm {
    fe delta, g_coset;                  // delta = Fr::DELTA; beta_zeta = beta * g_coset
    uint32_t n_cols, chunk_len, n_sets;
    int last_rot;                       // -(blinding_factors + 1)
    const fe *z;                        // n_sets columns per proof
    size_t z_stride, z_pstride;
    const fe *l0, *l_last, *l_active;
    const fe *tw;                       // extended_omega^i, i < n_ext / 2
    // a call may cover only the sets [set_begin, set_end) (the caller streams the extended columns through HBM in
    // slices, k = 20 proofs); `head` = fold the terms that precede the per-set products; the column tables then
    // start at column set_begin * chunk_len and delta_begin = delta^(set_begin * chunk_len)
    uint32_t set_begin, set_end, head;
    fe delta_begin;
};

template <class CC, class SC>
__global__ void __launch_bounds__(256) quotient_permutation_kernel(QuotientGroup g, QuotientCommon c, QuotientPerm p, CC cs, SC ss) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x, pr = blockIdx.y;
    if (idx >= c.n_ext) return;
    const CC cols = cs.at(pr);
    const SC sigma = ss.at(pr);
    fe *h = g.h + pr * g.h_stride;
    const fe *z = p.z + pr * p.z_pstride;
    const fe y = fe_load_global(g.scal + 3 * pr), beta = fe_load_global(g.scal + 3 * pr + 1), gamma = fe_load_global(g.scal + 3 * pr + 2);
    const uint32_t r_next = q_rot(idx, 1, c), r_last = q_rot(idx, p.last_rot, c);
    const fe one = fe_one<FrQ>();
    const fe l0 = fe_load_global(p.l0 + idx), l_last = fe_load_global(p.l_last + idx), l_active = fe_load_global(p.l_active + idx);
    fe v = fe_load_global(h + idx);
    if (p.head) {
        // l_0 * (1 - z_0)
        {
            fe z0 = fe_load_global(z + idx);
            v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(one, z0), l0));
        }
        // l_last * (z_l^2 - z_l)
        {
            fe zl = fe_load_global(z + (size_t)(p.n_sets - 1) * p.z_stride + idx);
            v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(fe_sqr<FrQ>(zl), zl), l_last));
        }
        // l_0 * (z_i - z_{i-1}(w^last X)),  i >= 1
        for (uint32_t s = 1; s < p.n_sets; ++s) {
            fe zi = fe_load_global(z + (size_t)s * p.z_stride + idx);
            fe zp = fe_load_global(z + (size_t)(s - 1) * p.z_stride + r_last);
            v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(zi, zp), l0));
        }
    }
    // l_active * ( z_i(wX) prod (v + beta sigma + gamma) - z_i(X) prod (v + delta^j beta X + gamma) )
    const uint32_t half = c.n_ext >> 1;
    fe w = fe_load_ro(p.tw + (idx & (half - 1)));
    if (idx >= half) w = fe_neg<FrQ>(w);
    fe cur = fe_mul<FrQ>(fe_mul<FrQ>(beta, p.g_coset), w);
    if (p.set_begin) cur = fe_mul<FrQ>(cur, p.delta_begin);
    const uint32_t col_base = p.set_begin * p.chunk_len;
    for (uint32_t s = p.set_begin; s < p.set_end; ++s) {
        const uint32_t c0 = s * p.chunk_len, c1 = min(c0 + p.chunk_len, p.n_cols);
        fe left = fe_load_global(z + (size_t)s * p.z_stride + r_next);
        fe right = fe_load_global(z + (size_t)s * p.z_stride + idx);
        for (uint32_t j = c0; j < c1; ++j) {
            fe val = fe_add<FrQ>(fe_load_global(cols.col(j - col_base) + idx), gamma);
            fe sg = fe_mul<FrQ>(beta, fe_load_global(sigma.col(j - col_base) + idx));
            left = fe_mul<FrQ>(left, fe_add<FrQ>(val, sg));
            right = fe_mul<FrQ>(right, fe_add<FrQ>(val, cur));
            cur = fe_mul<FrQ>(cur, p.delta);
        }
        v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(left, right), l_active));
    }
    fe_store_global(h + idx, v);
}

// lookup arguments: `n_lookups` of them per proof, folded in order; lookup l of proof p reads the five columns
// tab[p * pstride + 5 l + (0 .. 4)] = compressed input, compressed table (theta-folded by the caller), A', S', z
struct QuotientLookup {
    const fe *const *tab;
    size_t pstride;
    uint32_t n_lookups;
    const fe *l0, *l_last, *l_active;
};

__global__ void __launch_bounds__(256) quotient_lookup_kernel(QuotientGroup g, QuotientCommon c, QuotientLookup p) {
    const uint32_t idx = blockIdx.x * blockDim.x + threadIdx.x, pr = blockIdx.y;
    if (idx >= c.n_ext) return;
    fe *h = g.h + pr * g.h_stride;
    const fe y = fe_load_global(g.scal + 3 * pr), beta = fe_load_global(g.scal + 3 * pr + 1), gamma = fe_load_global(g.scal + 3 * pr + 2);
    const uint32_t r_next = q_rot(idx, 1, c), r_prev = q_rot(idx, -1, c);
    const fe one = fe_one<FrQ>();
    const fe l0 = fe_load_global(p.l0 + idx), l_last = fe_load_global(p.l_last + idx), l_active = fe_load_global(p.l_active + idx);
    fe v = fe_load_global(h + idx);
    for (uint32_t l = 0; l < p.n_lookups; ++l) {
        const fe *const *t = p.tab + pr * p.pstride + 5 * (size_t)l;
        const fe *input = t[0], *table = t[1], *perm_input = t[2], *perm_table = t[3], *zc = t[4];
        const fe z = fe_load_global(zc + idx), zn = fe_load_global(zc + r_next);
        const fe ap = fe_load_global(perm_input + idx), sp = fe_load_global(perm_table + idx);
        const fe a_minus_s = fe_sub<FrQ>(ap, sp);
        // l_0 * (1 - z)
        v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(one, z), l0));
        // l_last * (z^2 - z)
        v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(fe_sqr<FrQ>(z), z), l_last));
        // l_active * ( z(wX) (a' + beta)(s' + gamma) - z (a + beta)(s + gamma) )
        {
            fe left = fe_mul<FrQ>(fe_mul<FrQ>(zn, fe_add<FrQ>(ap, beta)), fe_add<FrQ>(sp, gamma));
            fe tv = fe_mul<FrQ>(fe_add<FrQ>(fe_load_global(input + idx), beta), fe_add<FrQ>(fe_load_global(table + idx), gamma));
            fe right = fe_mul<FrQ>(z, tv);
            v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_sub<FrQ>(left, right), l_active));
        }
        // l_0 * (a' - s')
        v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(a_minus_s, l0));
        // l_active * (a' - s') (a' - a'(w^-1 X))
        {
            fe d = fe_sub<FrQ>(ap, fe_load_global(perm_input + r_prev));
            v = fe_add<FrQ>(fe_mul<FrQ>(v, y), fe_mul<FrQ>(fe_mul<FrQ>(a_minus_s, d), l_active));
        }
    }
    fe_store_global(h + idx, v);
}

}  // namespace h2v
