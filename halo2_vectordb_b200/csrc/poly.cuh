// poly.cuh -- Fr polynomial primitives on either side of every commit ("next" row 2 of SURVEY.md 8(f)).
//
// Device counterparts of halo2-axiom arithmetic.rs `eval_polynomial` and `kate_division`,
// ff `BatchInvert::batch_invert`, and the running product z of plonk/permutation/prover.rs and
// plonk/lookup/prover.rs (z[0] = 1, z[i+1] = z[i] * num[i] / den[i]); all reached from
// /root/reference/src/scaffold/mod.rs:296 through create_proof (SURVEY.md 3.1 steps 6, 7, 12, 13).
// Every output is a uniquely determined vector of field elements, compared bit for bit with the oracle.
#pragma once
#include "ff.cuh"

namespace h2v {

typedef FrP Fr;

__device__ __forceinline__ fe pl_ld(const fe *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = q[0], b = q[1];
    fe r;
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    return r;
}
__device__ __forceinline__ void pl_st(fe *p, const fe &x) {
    uint4 *q = reinterpret_cast<uint4 *>(p);
    q[0] = make_uint4(x.v[0], x.v[1], x.v[2], x.v[3]);
    q[1] = make_uint4(x.v[4], x.v[5], x.v[6], x.v[7]);
}
__device__ __forceinline__ fe fe_shfl_up(const fe &v, int off) {
    fe r;
#pragma unroll
    for (int k = 0; k < 8; ++k) r.v[k] = __shfl_up_sync(0xffffffffu, v.v[k], off);
    return r;
}
__device__ __forceinline__ fe fe_shfl_down(const fe &v, int off) {
    fe r;
#pragma unroll
    for (int k = 0; k < 8; ++k) r.v[k] = __shfl_down_sync(0xffffffffu, v.v[k], off);
    return r;
}

struct OpMul {
    static __device__ __forceinline__ fe id() { return fe_one<Fr>(); }
    static __device__ __forceinline__ fe op(const fe &a, const fe &b) { return fe_mul<Fr>(a, b); }
};
struct OpAdd {
    static __device__ __forceinline__ fe id() { return fe_zero(); }
    static __device__ __forceinline__ fe op(const fe &a, const fe &b) { return fe_add<Fr>(a, b); }
};
// exclusive scan of one value per thread over a 256-thread CTA; *total = combination of all 256
template <class Op> __device__ __forceinline__ fe block_excl_scan_256(fe v, fe *total, fe *sm8) {
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    fe inc = v;
#pragma unroll 1
    for (int o = 1; o < 32; o <<= 1) {
        fe t = fe_shfl_up(inc, o);
        if ((int)lane >= o) inc = Op::op(t, inc);
    }
    fe exc = fe_shfl_up(inc, 1);
    if (lane == 0) exc = Op::id();
    __syncthreads();
    if (lane == 31) sm8[wid] = inc;
    __syncthreads();
    fe base = Op::id(), tot = Op::id();
#pragma unroll 1
    for (uint32_t w = 0; w < 8; ++w) {
        fe x = sm8[w];
        if (w < wid) base = Op::op(base, x);
        tot = Op::op(tot, x);
    }
    *total = tot;
    return Op::op(base, exc);
}

// ------------------------------------------------------------------ eval_polynomial
// out[poly * n_points + pt] = sum_i polys[poly][i] * x_pt^i.  grid (n_points, n_polys), 256 threads:
// each thread runs Horner over a contiguous slice, the slices are recombined with x^(slice start).
__global__ void __launch_bounds__(256) poly_eval_kernel(const fe *__restrict__ polys, size_t stride, uint32_t len,
                                                        const fe *__restrict__ points, uint32_t n_points, fe *__restrict__ out) {
    __shared__ fe sm8[8];
    const fe *a = polys + (size_t)blockIdx.y * stride;
    const fe x = pl_ld(points + blockIdx.x);
    const uint32_t chunk = (len + 255) / 256;
    const uint32_t lo = min(threadIdx.x * chunk, len), hi = min(lo + chunk, len);
    fe v = fe_zero();
    for (uint32_t i = hi; i-- > lo;) v = fe_add<Fr>(fe_mul<Fr>(v, x), pl_ld(a + i));
    // weight x^lo = (x^chunk)^tid
    fe w = fe_pow_small<Fr>(fe_pow_small<Fr>(x, chunk), threadIdx.x);
    v = fe_mul<Fr>(v, w);
#pragma unroll 1
    for (int o = 16; o >= 1; o >>= 1) v = fe_add<Fr>(v, fe_shfl_down(v, o));
    if ((threadIdx.x & 31) == 0) sm8[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        fe s = sm8[0];
        for (int wv = 1; wv < 8; ++wv) s = fe_add<Fr>(s, sm8[wv]);
        pl_st(out + (size_t)blockIdx.y * n_points + blockIdx.x, s);
    }
}

// ------------------------------------------------------------------ batch inversion: radix-G product tree, ONE field inversion at the root (all elements non-zero)
// P[i] = product of X[j] for j < i inside i's group of G;  Xn[g] = product of group g
template <class F> __global__ void __launch_bounds__(128) binv_up_kernel(const fe *__restrict__ X, fe *__restrict__ P, fe *__restrict__ Xn, uint32_t n, uint32_t G) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t lo = (uint64_t)g * G;
    if (lo >= n) return;
    uint32_t hi = (uint32_t)min((uint64_t)n, lo + G);
    fe run = fe_one<F>();
    for (uint32_t i = (uint32_t)lo; i < hi; ++i) {
        pl_st(P + i, run);
        run = fe_mul<F>(run, pl_ld(X + i));
    }
    pl_st(Xn + g, run);
}
template <class F> __global__ void binv_top_kernel(const fe *__restrict__ X, fe *__restrict__ I) {
    if (blockIdx.x == 0 && threadIdx.x == 0) pl_st(I, fe_inv_fast<F>(pl_ld(X)));
}
// I[i] = 1 / X[i] from In[g] = 1 / (product of group g)
template <class F> __global__ void __launch_bounds__(128) binv_down_kernel(const fe *__restrict__ X, const fe *__restrict__ P, const fe *__restrict__ In,
                                                        fe *__restrict__ I, uint32_t n, uint32_t G) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t lo = (uint64_t)g * G;
    if (lo >= n) return;
    uint32_t hi = (uint32_t)min((uint64_t)n, lo + G);
    fe inv = pl_ld(In + g);
    for (uint32_t i = hi; i-- > (uint32_t)lo;) {
        pl_st(I + i, fe_mul<F>(inv, pl_ld(P + i)));
        inv = fe_mul<F>(inv, pl_ld(X + i));
    }
}

// ------------------------------------------------------------------ batch inversion helpers: zeros are skipped as ff::BatchInvert does
__global__ void __launch_bounds__(256) fr_zero_to_one_kernel(const fe *__restrict__ a, fe *__restrict__ x, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe v = pl_ld(a + i);
    pl_st(x + i, fe_is_zero(v) ? fe_one<Fr>() : v);
}
__global__ void __launch_bounds__(256) fr_select_inverse_kernel(const fe *__restrict__ a, const fe *__restrict__ inv, fe *__restrict__ out, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe v = pl_ld(a + i);
    pl_st(out + i, fe_is_zero(v) ? v : pl_ld(inv + i));
}

// ------------------------------------------------------------------ running product
// r[i] = num[i] * dinv[i];  out[i] = product of r[j], j < i   (exclusive; out[0] = 1).  Tiles of 2048.
#define H2V_FR_TILE 2048
__global__ void __launch_bounds__(256) fr_prod_tiles_kernel(const fe *__restrict__ num, const fe *__restrict__ dinv, uint32_t n,
                                                            fe *__restrict__ tile_prod) {
    __shared__ fe sm8[8];
    // grid.y = column: columns are n elements apart, their tile products gridDim.x apart
    num += (size_t)blockIdx.y * n;
    dinv += (size_t)blockIdx.y * n;
    tile_prod += (size_t)blockIdx.y * gridDim.x;
    const uint32_t base = blockIdx.x * H2V_FR_TILE + threadIdx.x * 8;
    fe p = fe_one<Fr>();
#pragma unroll 1
    for (int k = 0; k < 8; ++k)
        if (base + k < n) p = fe_mul<Fr>(p, fe_mul<Fr>(pl_ld(num + base + k), pl_ld(dinv + base + k)));
    fe tot;
    block_excl_scan_256<OpMul>(p, &tot, sm8);
    if (threadIdx.x == 0) pl_st(tile_prod + blockIdx.x, tot);
}
// in-place exclusive scan of tile[0..ntiles) by one CTA (grid.y = column, `ntiles` apart)
template <class Op> __global__ void __launch_bounds__(256) fr_scan_top_kernel(fe *__restrict__ tile, uint32_t ntiles) {
    __shared__ fe sm8[8];
    tile += (size_t)blockIdx.y * ntiles;
    const uint32_t per = (ntiles + 255) / 256;
    const uint32_t lo = min(threadIdx.x * per, ntiles), hi = min(lo + per, ntiles);
    fe s = Op::id();
    for (uint32_t k = lo; k < hi; ++k) s = Op::op(s, pl_ld(tile + k));
    fe tot;
    fe run = block_excl_scan_256<Op>(s, &tot, sm8);
    for (uint32_t k = lo; k < hi; ++k) {
        fe v = pl_ld(tile + k);
        pl_st(tile + k, run);
        run = Op::op(run, v);
    }
}
__global__ void __launch_bounds__(256) fr_prod_apply_kernel(const fe *__restrict__ num, const fe *__restrict__ dinv, uint32_t n,
                                                            const fe *__restrict__ tile_pre, fe *__restrict__ out) {
    __shared__ fe sm8[8];
    num += (size_t)blockIdx.y * n;
    dinv += (size_t)blockIdx.y * n;
    out += (size_t)blockIdx.y * n;
    tile_pre += (size_t)blockIdx.y * gridDim.x;
    const uint32_t base = blockIdx.x * H2V_FR_TILE + threadIdx.x * 8;
    fe r[8];
    fe p = fe_one<Fr>();
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        r[k] = (base + k < n) ? fe_mul<Fr>(pl_ld(num + base + k), pl_ld(dinv + base + k)) : fe_one<Fr>();
        p = fe_mul<Fr>(p, r[k]);
    }
    fe tot;
    fe run = fe_mul<Fr>(block_excl_scan_256<OpMul>(p, &tot, sm8), pl_ld(tile_pre + blockIdx.x));
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        if (base + k < n) pl_st(out + base + k, run);
        run = fe_mul<Fr>(run, r[k]);
    }
}

// ------------------------------------------------------------------ kate_division
// Many columns at once (grid.y = column), each with its own length and point: column j divides a[0 .. n) by (X - b)
// into q[0 .. n - 1).  q[i] = b^-(i+1) * S[i+1],  S[k] = sum_{j >= k} a[j] b^j  (b != 0).  Forward index k <-> j = n-1-k:
// t_k = a[n-1-k] b^(n-1-k), inclusive prefix sums P_k = S[n-1-k], q[n-2-k] = P_k * binv^(n-1-k).  b == 0: q[i] = a[i+1].
// The tile sums of column j lie at tile + j * ntiles (ntiles covers the longest column).
struct KateCol {
    const fe *a;
    fe *q;
    uint32_t n;
    fe b, binv;      // binv: unused when b == 0
};
__device__ __forceinline__ void kate_thread(const KateCol &p, uint32_t base, fe (&t)[8], fe &sum) {
    // powers b^(n-1-base), then multiply by binv per step
    fe pw = (base < p.n) ? fe_pow_small<Fr>(p.b, p.n - 1 - base) : fe_zero();
    sum = fe_zero();
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        if (base + k < p.n) {
            t[k] = fe_mul<Fr>(pl_ld(p.a + (p.n - 1 - base - k)), pw);
            pw = fe_mul<Fr>(pw, p.binv);
        } else {
            t[k] = fe_zero();
        }
        sum = fe_add<Fr>(sum, t[k]);
    }
}
__global__ void __launch_bounds__(256) kate_tiles_kernel(const KateCol *cols, fe *tile, uint32_t ntiles) {
    __shared__ fe sm8[8];
    const KateCol p = cols[blockIdx.y];
    if (fe_is_zero(p.b)) return;          // the shift needs no tile sums (uniform over the CTA)
    fe t[8], s, tot;
    kate_thread(p, blockIdx.x * H2V_FR_TILE + threadIdx.x * 8, t, s);
    block_excl_scan_256<OpAdd>(s, &tot, sm8);
    if (threadIdx.x == 0) pl_st(tile + (size_t)blockIdx.y * ntiles + blockIdx.x, tot);
}
__global__ void __launch_bounds__(256) kate_apply_kernel(const KateCol *cols, const fe *tile, uint32_t ntiles) {
    __shared__ fe sm8[8];
    const KateCol p = cols[blockIdx.y];
    const uint32_t base = blockIdx.x * H2V_FR_TILE + threadIdx.x * 8;
    if (fe_is_zero(p.b)) {
        for (uint32_t i = base; i < base + 8; ++i)
            if (i + 1 < p.n) pl_st(p.q + i, pl_ld(p.a + i + 1));
        return;
    }
    fe t[8], s, tot;
    kate_thread(p, base, t, s);
    fe run = fe_add<Fr>(block_excl_scan_256<OpAdd>(s, &tot, sm8), pl_ld(tile + (size_t)blockIdx.y * ntiles + blockIdx.x));
    // output factor binv^(n-1-k), stepping up by b
    fe f = (base < p.n) ? fe_pow_small<Fr>(p.binv, p.n - 1 - base) : fe_zero();
#pragma unroll 1
    for (int k = 0; k < 8; ++k) {
        const uint32_t kk = base + k;
        run = fe_add<Fr>(run, t[k]);                 // inclusive prefix P_kk
        if (kk + 1 < p.n) pl_st(p.q + (p.n - 2 - kk), fe_mul<Fr>(run, f));
        f = fe_mul<Fr>(f, p.b);
    }
}

}  // namespace h2v
