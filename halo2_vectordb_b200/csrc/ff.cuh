// ff.cuh -- BN254 Fr / Fq arithmetic, 8 x 32-bit limbs, Montgomery form (R = 2^256).
//
// Replaces (device side) halo2curves bn256::{Fr,Fq} `mul/add/sub/neg/square/invert`
// (SURVEY.md 8(a) row a13; reached from /root/reference/src/scaffold/mod.rs:273,296).
// Memory layout is byte-identical to halo2curves' `[u64;4]` little-endian Montgomery limbs, so
// host slices cross the C ABI without conversion.
//
// Device path: interleaved (CIOS) Montgomery product on two accumulators -- one holding the
// products of the even limbs of `a`, one the odd limbs, the second offset by 32 bits -- so every
// 64-bit partial product lands on an aligned limb pair and a whole row is one carry chain of
// mad.lo.cc / madc.hi.cc pairs, which ptxas fuses into IMAD.WIDE.U32(.X) on sm_100a.
// 8*16 wide multiply-adds + 8 low multiplies (the Montgomery quotients) = 136 per product, plus three adds per row
// (the stray limb and the two carries that land directly in the top limb) -- the SASS of a product is a straight
// stream of IMAD.WIDE.U32.X.  Lazily reduced variants (fe_mul_lazy, fe_sub_lazy, fe_csub_2m ...) serve the NTT
// butterflies and the MSM accumulation loop, which keep values in [0, 4m) / [0, 2m) between products.
// Host path (same file, !__CUDA_ARCH__): portable u64 arithmetic, used for domain constants and
// by the host-side unit checks.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define H2V_HD __host__ __device__ __forceinline__
#else
#define H2V_HD inline
#endif

namespace h2v {

struct alignas(16) fe {
    uint32_t v[8];
};

// ------------------------------------------------------------------ field parameters
// SURVEY.md App. B; re-derived in oracle/pyref.py, checked by tests/test_oracle.py::test_constants
struct FqP {
    static H2V_HD uint32_t m(int i) {
        return i == 0 ? 0xd87cfd47u : i == 1 ? 0x3c208c16u : i == 2 ? 0x6871ca8du : i == 3 ? 0x97816a91u
             : i == 4 ? 0x8181585du : i == 5 ? 0xb85045b6u : i == 6 ? 0xe131a029u : 0x30644e72u;
    }
    static H2V_HD uint32_t inv() { return 0xe4866389u; }   // -p^{-1} mod 2^32
    static H2V_HD uint32_t r1(int i) {                      // R mod p
        return i == 0 ? 0xc58f0d9du : i == 1 ? 0xd35d438du : i == 2 ? 0xf5c70b3du : i == 3 ? 0x0a78eb28u
             : i == 4 ? 0x7879462cu : i == 5 ? 0x666ea36fu : i == 6 ? 0x9a07df2fu : 0x0e0a77c1u;
    }
    static H2V_HD uint32_t r2(int i) {                      // R^2 mod p
        return i == 0 ? 0x538afa89u : i == 1 ? 0xf32cfc5bu : i == 2 ? 0xd44501fbu : i == 3 ? 0xb5e71911u
             : i == 4 ? 0x0a417ff6u : i == 5 ? 0x47ab1effu : i == 6 ? 0xcab8351fu : 0x06d89f71u;
    }
    static H2V_HD uint32_t r3(int i) {                      // R^3 mod p
        return i == 0 ? 0xda1530dfu : i == 1 ? 0xb1cd6dafu : i == 2 ? 0xa7283db6u : i == 3 ? 0x62f210e6u
             : i == 4 ? 0x0ada0afbu : i == 5 ? 0xef7f0b0cu : i == 6 ? 0x2d592544u : 0x20fd6e90u;
    }
};
struct FrP {
    static H2V_HD uint32_t m(int i) {
        return i == 0 ? 0xf0000001u : i == 1 ? 0x43e1f593u : i == 2 ? 0x79b97091u : i == 3 ? 0x2833e848u
             : i == 4 ? 0x8181585du : i == 5 ? 0xb85045b6u : i == 6 ? 0xe131a029u : 0x30644e72u;
    }
    static H2V_HD uint32_t inv() { return 0xefffffffu; }   // -r^{-1} mod 2^32
    static H2V_HD uint32_t r1(int i) {
        return i == 0 ? 0x4ffffffbu : i == 1 ? 0xac96341cu : i == 2 ? 0x9f60cd29u : i == 3 ? 0x36fc7695u
             : i == 4 ? 0x7879462eu : i == 5 ? 0x666ea36fu : i == 6 ? 0x9a07df2fu : 0x0e0a77c1u;
    }
    static H2V_HD uint32_t r2(int i) {
        return i == 0 ? 0xae216da7u : i == 1 ? 0x1bb8e645u : i == 2 ? 0xe35c59e3u : i == 3 ? 0x53fe3ab1u
             : i == 4 ? 0x53bb8085u : i == 5 ? 0x8c49833du : i == 6 ? 0x7f4e44a5u : 0x0216d0b1u;
    }
    static H2V_HD uint32_t r3(int i) {
        return i == 0 ? 0xb4bf0040u : i == 1 ? 0x5e94d8e1u : i == 2 ? 0x1cfbb6b8u : i == 3 ? 0x2a489cbeu
             : i == 4 ? 0xa19fcfedu : i == 5 ? 0x893cc664u : i == 6 ? 0x7fcc657cu : 0x0cf8594bu;
    }
};

// ------------------------------------------------------------------ small helpers
H2V_HD fe fe_zero() {
    fe r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = 0;
    return r;
}
template <class F> H2V_HD fe fe_one() {
    fe r;
#pragma unroll
    for (int i = 0; i < 8; ++i) r.v[i] = F::r1(i);
    return r;
}
H2V_HD bool fe_is_zero(const fe &a) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a.v[i];
    return o == 0;
}
H2V_HD bool fe_eq(const fe &a, const fe &b) {
    uint32_t o = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) o |= a.v[i] ^ b.v[i];
    return o == 0;
}
#ifdef __CUDACC__
// order and equality of sort keys (canonical integers, 8 limbs)
__device__ __forceinline__ bool key_less(const fe &a, const fe &b) {
#pragma unroll
    for (int i = 7; i >= 0; --i)
        if (a.v[i] != b.v[i]) return a.v[i] < b.v[i];
    return false;
}
__device__ __forceinline__ bool key_eq(const fe &a, const fe &b) {
    uint32_t d = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) d |= a.v[i] ^ b.v[i];
    return d == 0;
}
#endif

// ------------------------------------------------------------------ add / sub
#ifdef __CUDA_ARCH__
// r = a + b (no reduction); both < 2^255 so no carry out of limb 7
__device__ __forceinline__ void raw_add(uint32_t *r, const uint32_t *a, const uint32_t *b) {
    asm("add.cc.u32 %0, %8, %16;\n\t"
        "addc.cc.u32 %1, %9, %17;\n\t"
        "addc.cc.u32 %2, %10, %18;\n\t"
        "addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\t"
        "addc.cc.u32 %5, %13, %21;\n\t"
        "addc.cc.u32 %6, %14, %22;\n\t"
        "addc.u32 %7, %15, %23;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
}
// r = a - b, returns borrow mask (0xffffffff if a < b)
__device__ __forceinline__ uint32_t raw_sub(uint32_t *r, const uint32_t *a, const uint32_t *b) {
    uint32_t bw;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(bw)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
          "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    return bw;
}
#else
inline void raw_add(uint32_t *r, const uint32_t *a, const uint32_t *b) {
    uint64_t c = 0;
    for (int i = 0; i < 8; ++i) {
        c += (uint64_t)a[i] + b[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
}
inline uint32_t raw_sub(uint32_t *r, const uint32_t *a, const uint32_t *b) {
    uint64_t bw = 0;
    for (int i = 0; i < 8; ++i) {
        uint64_t d = (uint64_t)a[i] - b[i] - bw;
        r[i] = (uint32_t)d;
        bw = (d >> 32) & 1;
    }
    return bw ? 0xffffffffu : 0u;
}
#endif

// if t >= m: t -= m   (t < 2m on entry)
template <class F> H2V_HD void fe_reduce_once(fe &t) {
    uint32_t mm[8], d[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = F::m(i);
    uint32_t bw = raw_sub(d, t.v, mm);
#pragma unroll
    for (int i = 0; i < 8; ++i) t.v[i] = bw ? t.v[i] : d[i];
}
template <class F> H2V_HD fe fe_add(const fe &a, const fe &b) {
    fe r;
    raw_add(r.v, a.v, b.v);
    fe_reduce_once<F>(r);
    return r;
}
template <class F> H2V_HD fe fe_sub(const fe &a, const fe &b) {
    fe r;
    uint32_t bw = raw_sub(r.v, a.v, b.v);
    if (bw) {      // predicated add of m (no masks)
        uint32_t mm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) mm[i] = F::m(i);
        raw_add(r.v, r.v, mm);
    }
    return r;
}
template <class F> H2V_HD fe fe_neg(const fe &a) {
    if (fe_is_zero(a)) return a;
    fe r;
    uint32_t mm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = F::m(i);
    raw_sub(r.v, mm, a.v);
    return r;
}
template <class F> H2V_HD fe fe_dbl(const fe &a) { return fe_add<F>(a, a); }

// ------------------------------------------------------------------ Montgomery product
#ifdef __CUDA_ARCH__
// acc[0..7] = sum_t (x[2t] * y) << (64 t)            (four independent 64-bit products)
__device__ __forceinline__ void row_mul(uint32_t *acc, const uint32_t *x, uint32_t y) {
    // one IMAD.WIDE.U32 per product (a mul.lo / mul.hi pair is NOT fused by ptxas: two multiplier-pipe instructions)
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const uint64_t p = (uint64_t)x[2 * t] * y;
        acc[2 * t] = (uint32_t)p;
        acc[2 * t + 1] = (uint32_t)(p >> 32);
    }
}
// acc[0..7] += sum_t (x[2t] * y) << (64 t); returns the carry out of limb 7 (0 or 1)
__device__ __forceinline__ uint32_t row_mad(uint32_t *acc, const uint32_t *x, uint32_t y) {
    uint32_t c;
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=&r"(c)
        : "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(y));
    return c;
}
// acc[0..7] += sum_t (x[2t] * y) << (64 t), the carry out of limb 7 goes straight into `top` (one instruction
// instead of a carry capture plus an add)
__device__ __forceinline__ void row_mad_top(uint32_t *acc, const uint32_t *x, uint32_t y, uint32_t &top) {
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
        : "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(y));
}
// Shift-and-accumulate for the offset accumulator when its partner drops one limb:
//   lo0 += stray (carry c0);  out[0..7] = {in[2..7],0,0} + sum_t (x[2t] * y) << (64 t) + c0
__device__ __forceinline__ void row_mad_shift(uint32_t *out, const uint32_t *in, uint32_t &lo0, uint32_t stray,
                                              const uint32_t *x, uint32_t y) {
    asm("add.cc.u32 %8, %8, %9;\n\t"
        "madc.lo.cc.u32 %0, %10, %14, %15;\n\t"
        "madc.hi.cc.u32 %1, %10, %14, %16;\n\t"
        "madc.lo.cc.u32 %2, %11, %14, %17;\n\t"
        "madc.hi.cc.u32 %3, %11, %14, %18;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %19;\n\t"
        "madc.hi.cc.u32 %5, %12, %14, %20;\n\t"
        "madc.lo.cc.u32 %6, %13, %14, 0;\n\t"
        "madc.hi.u32 %7, %13, %14, 0;"
        : "=&r"(out[0]), "=&r"(out[1]), "=&r"(out[2]), "=&r"(out[3]), "=&r"(out[4]), "=&r"(out[5]), "=&r"(out[6]), "=&r"(out[7]),
          "+r"(lo0)
        : "r"(stray), "r"(x[0]), "r"(x[2]), "r"(x[4]), "r"(x[6]), "r"(y),
          "r"(in[2]), "r"(in[3]), "r"(in[4]), "r"(in[5]), "r"(in[6]), "r"(in[7]));
}

// One CIOS row.  On entry (FIRST == false): T = lo + hi * 2^32 with lo[0] == 0 from the previous
// reduction.  T <- (T >> 32) + a * bi, then T += q * m with q chosen so the low limb vanishes.
// The accumulators swap roles: new lo = old hi, new hi = old lo >> 64, old lo[1] is the stray limb.
template <class F, bool FIRST>
__device__ __forceinline__ void mont_row(uint32_t *lo, uint32_t *hi, const uint32_t *a, uint32_t bi) {
    // (lo, hi) are the accumulators in their roles for THIS row (caller swaps them every row).
    uint32_t mm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = F::m(i);
    if (FIRST) {
        row_mul(lo, a, bi);
        row_mul(hi, a + 1, bi);
    } else {
        // on entry `hi` holds the OLD low accumulator (limb 0 is zero, limb 1 is the stray) and `lo` the old high one
        uint32_t nh[8];
        row_mad_shift(nh, hi, lo[0], hi[1], a + 1, bi);
#pragma unroll
        for (int i = 0; i < 8; ++i) hi[i] = nh[i];
        row_mad_top(lo, a, bi, hi[7]);
    }
    uint32_t q = lo[0] * F::inv();
    row_mad(hi, mm + 1, q);              // cannot carry out: T < 2 * 2^32 * m < 2^288
    row_mad_top(lo, mm, q, hi[7]);
}

// Montgomery product without the final conditional subtraction: a * b / R + (< m).  For a < 4m and b < m the result
// is < 2m (4m^2 / R + m = 1.76 m for both BN254 fields) and every intermediate stays below 2^288.
template <class F> __device__ __forceinline__ fe fe_mul_lazy(const fe &a, const fe &b) {
    uint32_t e[8], o[8];
    mont_row<F, true>(e, o, a.v, b.v[0]);
    mont_row<F, false>(o, e, a.v, b.v[1]);
    mont_row<F, false>(e, o, a.v, b.v[2]);
    mont_row<F, false>(o, e, a.v, b.v[3]);
    mont_row<F, false>(e, o, a.v, b.v[4]);
    mont_row<F, false>(o, e, a.v, b.v[5]);
    mont_row<F, false>(e, o, a.v, b.v[6]);
    mont_row<F, false>(o, e, a.v, b.v[7]);
    // after 8 rows: low accumulator = o (o[0] == 0), high = e.  result = e + (o >> 32)
    fe r;
    asm("add.cc.u32 %0, %8, %16;\n\t"
        "addc.cc.u32 %1, %9, %17;\n\t"
        "addc.cc.u32 %2, %10, %18;\n\t"
        "addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\t"
        "addc.cc.u32 %5, %13, %21;\n\t"
        "addc.cc.u32 %6, %14, %22;\n\t"
        "addc.u32 %7, %15, 0;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7])
        : "r"(e[0]), "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]),
          "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]));
    return r;
}
template <class F> __device__ __forceinline__ fe fe_mul(const fe &a, const fe &b) {
    fe r = fe_mul_lazy<F>(a, b);
    fe_reduce_once<F>(r);
    return r;
}

// ---- dedicated Montgomery squaring: 108 wide multiply-adds instead of 136.
// a^2 = 2 S + D with S the 28 products a_i a_j (i < j) and D the 8 squares a_i^2; the 512-bit T = 2 S + D is then
// reduced by eight CIOS rows that carry no partial product (the quotient digits only depend on the low half, so the
// rows run on a window seeded with T[0..8) whose top limbs are fresh, exactly like fe_mul_lazy's, and T[8..16) is
// added at the end).  S is accumulated on an even / odd accumulator pair like the product rows: E holds the products
// that land on an even limb, O (one limb up) those on an odd limb, so every row is one mad.lo.cc / madc.hi.cc chain.
// For a < 2m the result is below 4 m^2 / R + m + 1 <= 2m, as for fe_mul_lazy.
template <class F> __device__ __forceinline__ void red_row(uint32_t *lo, uint32_t *hi) {
    // fe_mul_lazy's mont_row<F, false> without its partial product: `hi` is the old low accumulator (limb 0 zero, limb 1
    // the stray), `lo` the old high one
    uint32_t mm[8], nh[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = F::m(i);
    asm("add.cc.u32 %8, %8, %9;\n\t"
        "addc.cc.u32 %0, %10, 0;\n\t"
        "addc.cc.u32 %1, %11, 0;\n\t"
        "addc.cc.u32 %2, %12, 0;\n\t"
        "addc.cc.u32 %3, %13, 0;\n\t"
        "addc.cc.u32 %4, %14, 0;\n\t"
        "addc.cc.u32 %5, %15, 0;\n\t"
        "addc.cc.u32 %6, 0, 0;\n\t"
        "addc.u32 %7, 0, 0;"
        : "=&r"(nh[0]), "=&r"(nh[1]), "=&r"(nh[2]), "=&r"(nh[3]), "=&r"(nh[4]), "=&r"(nh[5]), "=&r"(nh[6]), "=&r"(nh[7]), "+r"(lo[0])
        : "r"(hi[1]), "r"(hi[2]), "r"(hi[3]), "r"(hi[4]), "r"(hi[5]), "r"(hi[6]), "r"(hi[7]));
#pragma unroll
    for (int i = 0; i < 8; ++i) hi[i] = nh[i];
    uint32_t q = lo[0] * F::inv();
    row_mad(hi, mm + 1, q);
    row_mad_top(lo, mm, q, hi[7]);
}
template <class F> __device__ __forceinline__ fe fe_sqr_lazy(const fe &x) {
    const uint32_t *a = x.v;
    uint32_t E2, E3, E4, E5, E6, E7, E8, E9, E10, E11, E12, E13;
    uint32_t O[14];
    // row a0: E <- a0 * (a2, a4, a6) on limbs 2..7, O <- a0 * (a1, a3, a5, a7) on limbs 0..7 (fresh limbs: plain products)
    {
        const uint64_t p2 = (uint64_t)a[0] * a[2], p4 = (uint64_t)a[0] * a[4], p6 = (uint64_t)a[0] * a[6];
        E2 = (uint32_t)p2; E3 = (uint32_t)(p2 >> 32);
        E4 = (uint32_t)p4; E5 = (uint32_t)(p4 >> 32);
        E6 = (uint32_t)p6; E7 = (uint32_t)(p6 >> 32);
    }
    row_mul(O, a + 1, a[0]);
    // row a1: E += a1 * (a3, a5, a7) on limbs 4..9 (8, 9 fresh); O += a1 * (a2, a4, a6) on limbs 2..7, carry into 8
    asm("mad.lo.cc.u32 %0, %6, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %8, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %8, %3;\n\t"
        "madc.lo.cc.u32 %4, %6, %9, 0;\n\t"
        "madc.hi.u32 %5, %6, %9, 0;"
        : "+r"(E4), "+r"(E5), "+r"(E6), "+r"(E7), "=&r"(E8), "=&r"(E9)
        : "r"(a[1]), "r"(a[3]), "r"(a[5]), "r"(a[7]));
    asm("mad.lo.cc.u32 %0, %7, %8, %0;\n\t"
        "madc.hi.cc.u32 %1, %7, %8, %1;\n\t"
        "madc.lo.cc.u32 %2, %7, %9, %2;\n\t"
        "madc.hi.cc.u32 %3, %7, %9, %3;\n\t"
        "madc.lo.cc.u32 %4, %7, %10, %4;\n\t"
        "madc.hi.cc.u32 %5, %7, %10, %5;\n\t"
        "addc.u32 %6, 0, 0;"
        : "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]), "+r"(O[6]), "+r"(O[7]), "=&r"(O[8])
        : "r"(a[1]), "r"(a[2]), "r"(a[4]), "r"(a[6]));
    // row a2: E += a2 * (a4, a6) on limbs 6..9, carry into 10; O += a2 * (a3, a5, a7) on limbs 4..9 (9 fresh)
    asm("mad.lo.cc.u32 %0, %5, %6, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %6, %1;\n\t"
        "madc.lo.cc.u32 %2, %5, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %5, %7, %3;\n\t"
        "addc.u32 %4, 0, 0;"
        : "+r"(E6), "+r"(E7), "+r"(E8), "+r"(E9), "=&r"(E10)
        : "r"(a[2]), "r"(a[4]), "r"(a[6]));
    asm("mad.lo.cc.u32 %0, %6, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %8, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %8, %3;\n\t"
        "madc.lo.cc.u32 %4, %6, %9, %4;\n\t"
        "madc.hi.u32 %5, %6, %9, 0;"
        : "+r"(O[4]), "+r"(O[5]), "+r"(O[6]), "+r"(O[7]), "+r"(O[8]), "=&r"(O[9])
        : "r"(a[2]), "r"(a[3]), "r"(a[5]), "r"(a[7]));
    // row a3: E += a3 * (a5, a7) on limbs 8..11 (11 fresh); O += a3 * (a4, a6) on limbs 6..9, carry into 10
    asm("mad.lo.cc.u32 %0, %4, %5, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, %5, %1;\n\t"
        "madc.lo.cc.u32 %2, %4, %6, %2;\n\t"
        "madc.hi.u32 %3, %4, %6, 0;"
        : "+r"(E8), "+r"(E9), "+r"(E10), "=&r"(E11)
        : "r"(a[3]), "r"(a[5]), "r"(a[7]));
    asm("mad.lo.cc.u32 %0, %5, %6, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %6, %1;\n\t"
        "madc.lo.cc.u32 %2, %5, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %5, %7, %3;\n\t"
        "addc.u32 %4, 0, 0;"
        : "+r"(O[6]), "+r"(O[7]), "+r"(O[8]), "+r"(O[9]), "=&r"(O[10])
        : "r"(a[3]), "r"(a[4]), "r"(a[6]));
    // row a4: E += a4 * a6 on limbs 10..11, carry into 12; O += a4 * (a5, a7) on limbs 8..11 (11 fresh)
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, 0, 0;"
        : "+r"(E10), "+r"(E11), "=&r"(E12)
        : "r"(a[4]), "r"(a[6]));
    asm("mad.lo.cc.u32 %0, %4, %5, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, %5, %1;\n\t"
        "madc.lo.cc.u32 %2, %4, %6, %2;\n\t"
        "madc.hi.u32 %3, %4, %6, 0;"
        : "+r"(O[8]), "+r"(O[9]), "+r"(O[10]), "=&r"(O[11])
        : "r"(a[4]), "r"(a[5]), "r"(a[7]));
    // row a5: E += a5 * a7 on limbs 12..13 (13 fresh); O += a5 * a6 on limbs 10..11, carry into 12
    asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t"
        "madc.hi.u32 %1, %2, %3, 0;"
        : "+r"(E12), "=&r"(E13)
        : "r"(a[5]), "r"(a[7]));
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, 0, 0;"
        : "+r"(O[10]), "+r"(O[11]), "=&r"(O[12])
        : "r"(a[5]), "r"(a[6]));
    // row a6: O += a6 * a7 on limbs 12..13 (13 fresh)
    asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t"
        "madc.hi.u32 %1, %2, %3, 0;"
        : "+r"(O[12]), "=&r"(O[13])
        : "r"(a[6]), "r"(a[7]));
    // S = E + (O << 32): limbs 1..15 (limb 0 is zero)
    uint32_t S[16];
    S[0] = 0;
    S[1] = O[0];
    asm("add.cc.u32 %0, %14, %28;\n\t"
        "addc.cc.u32 %1, %15, %29;\n\t"
        "addc.cc.u32 %2, %16, %30;\n\t"
        "addc.cc.u32 %3, %17, %31;\n\t"
        "addc.cc.u32 %4, %18, %32;\n\t"
        "addc.cc.u32 %5, %19, %33;\n\t"
        "addc.cc.u32 %6, %20, %34;\n\t"
        "addc.cc.u32 %7, %21, %35;\n\t"
        "addc.cc.u32 %8, %22, %36;\n\t"
        "addc.cc.u32 %9, %23, %37;\n\t"
        "addc.cc.u32 %10, %24, %38;\n\t"
        "addc.cc.u32 %11, %25, %39;\n\t"
        "addc.cc.u32 %12, %26, 0;\n\t"
        "addc.u32 %13, 0, 0;"
        : "=&r"(S[2]), "=&r"(S[3]), "=&r"(S[4]), "=&r"(S[5]), "=&r"(S[6]), "=&r"(S[7]), "=&r"(S[8]), "=&r"(S[9]), "=&r"(S[10]),
          "=&r"(S[11]), "=&r"(S[12]), "=&r"(S[13]), "=&r"(S[14]), "=&r"(S[15])
        : "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]), "r"(O[8]), "r"(O[9]), "r"(O[10]), "r"(O[11]),
          "r"(O[12]), "r"(O[13]), "r"(0u),
          "r"(E2), "r"(E3), "r"(E4), "r"(E5), "r"(E6), "r"(E7), "r"(E8), "r"(E9), "r"(E10), "r"(E11), "r"(E12), "r"(E13));
    // T = 2 S + D
    uint32_t T[16];
    T[0] = 0;
#pragma unroll
    for (int k = 1; k < 16; ++k) T[k] = __funnelshift_l(S[k - 1], S[k], 1);
    asm("mad.lo.cc.u32 %0, %16, %16, %0;\n\t"
        "madc.hi.cc.u32 %1, %16, %16, %1;\n\t"
        "madc.lo.cc.u32 %2, %17, %17, %2;\n\t"
        "madc.hi.cc.u32 %3, %17, %17, %3;\n\t"
        "madc.lo.cc.u32 %4, %18, %18, %4;\n\t"
        "madc.hi.cc.u32 %5, %18, %18, %5;\n\t"
        "madc.lo.cc.u32 %6, %19, %19, %6;\n\t"
        "madc.hi.cc.u32 %7, %19, %19, %7;\n\t"
        "madc.lo.cc.u32 %8, %20, %20, %8;\n\t"
        "madc.hi.cc.u32 %9, %20, %20, %9;\n\t"
        "madc.lo.cc.u32 %10, %21, %21, %10;\n\t"
        "madc.hi.cc.u32 %11, %21, %21, %11;\n\t"
        "madc.lo.cc.u32 %12, %22, %22, %12;\n\t"
        "madc.hi.cc.u32 %13, %22, %22, %13;\n\t"
        "madc.lo.cc.u32 %14, %23, %23, %14;\n\t"
        "madc.hi.u32 %15, %23, %23, %15;"
        : "+r"(T[0]), "+r"(T[1]), "+r"(T[2]), "+r"(T[3]), "+r"(T[4]), "+r"(T[5]), "+r"(T[6]), "+r"(T[7]), "+r"(T[8]), "+r"(T[9]),
          "+r"(T[10]), "+r"(T[11]), "+r"(T[12]), "+r"(T[13]), "+r"(T[14]), "+r"(T[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
    // Montgomery reduction of the low half
    uint32_t e[8], o[8], mm[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        e[i] = T[i];
        mm[i] = F::m(i);
    }
    {
        uint32_t q = e[0] * F::inv();
        row_mul(o, mm + 1, q);
        row_mad_top(e, mm, q, o[7]);
    }
    red_row<F>(o, e);
    red_row<F>(e, o);
    red_row<F>(o, e);
    red_row<F>(e, o);
    red_row<F>(o, e);
    red_row<F>(e, o);
    red_row<F>(o, e);
    // low accumulator = o (o[0] == 0), high = e: result = e + (o >> 32) + T[8..16)
    fe r;
    asm("add.cc.u32 %0, %8, %16;\n\t"
        "addc.cc.u32 %1, %9, %17;\n\t"
        "addc.cc.u32 %2, %10, %18;\n\t"
        "addc.cc.u32 %3, %11, %19;\n\t"
        "addc.cc.u32 %4, %12, %20;\n\t"
        "addc.cc.u32 %5, %13, %21;\n\t"
        "addc.cc.u32 %6, %14, %22;\n\t"
        "addc.u32 %7, %15, 0;"
        : "=&r"(r.v[0]), "=&r"(r.v[1]), "=&r"(r.v[2]), "=&r"(r.v[3]), "=&r"(r.v[4]), "=&r"(r.v[5]), "=&r"(r.v[6]), "=&r"(r.v[7])
        : "r"(e[0]), "r"(e[1]), "r"(e[2]), "r"(e[3]), "r"(e[4]), "r"(e[5]), "r"(e[6]), "r"(e[7]),
          "r"(o[1]), "r"(o[2]), "r"(o[3]), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]));
    fe hi_half;
#pragma unroll
    for (int i = 0; i < 8; ++i) hi_half.v[i] = T[8 + i];
    fe out;
    raw_add(out.v, r.v, hi_half.v);
    return out;
}
#else
template <class F> inline fe fe_mul(const fe &a, const fe &b) {
    uint32_t t[10] = {0};
    for (int i = 0; i < 8; ++i) {
        uint64_t c = 0;
        for (int j = 0; j < 8; ++j) {
            c += (uint64_t)a.v[j] * b.v[i] + t[j];
            t[j] = (uint32_t)c;
            c >>= 32;
        }
        c += t[8];
        t[8] = (uint32_t)c;
        t[9] = (uint32_t)(c >> 32);
        uint32_t q = t[0] * F::inv();
        c = (uint64_t)q * F::m(0) + t[0];
        c >>= 32;
        for (int j = 1; j < 8; ++j) {
            c += (uint64_t)q * F::m(j) + t[j];
            t[j - 1] = (uint32_t)c;
            c >>= 32;
        }
        c += t[8];
        t[7] = (uint32_t)c;
        t[8] = t[9] + (uint32_t)(c >> 32);
    }
    fe r;
    for (int i = 0; i < 8; ++i) r.v[i] = t[i];
    fe_reduce_once<F>(r);   // t[8] == 0 here because m < 2^254
    return r;
}
template <class F> inline fe fe_mul_lazy(const fe &a, const fe &b) { return fe_mul<F>(a, b); }   // host: always reduced
template <class F> inline fe fe_sqr_lazy(const fe &a) { return fe_mul<F>(a, a); }
#endif
// if t >= 2m: t -= 2m   (lazy-reduction helpers for the NTT butterflies: values live in [0, 4m), 4m < 2^256)
template <class F> H2V_HD uint32_t fe_2m_limb(int i) { return (F::m(i) << 1) | (i ? (F::m(i - 1) >> 31) : 0u); }
template <class F> H2V_HD void fe_csub_2m(fe &t) {
    uint32_t mm[8], d[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = fe_2m_limb<F>(i);
    uint32_t bw = raw_sub(d, t.v, mm);
#pragma unroll
    for (int i = 0; i < 8; ++i) t.v[i] = bw ? t.v[i] : d[i];
}
// a - b for a, b in [0, 2m), result in [0, 2m)
template <class F> H2V_HD fe fe_sub_lazy(const fe &a, const fe &b) {
    fe r;
    uint32_t bw = raw_sub(r.v, a.v, b.v);
    if (bw) {      // predicated add of 2m (no masks)
        uint32_t mm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) mm[i] = fe_2m_limb<F>(i);
        raw_add(r.v, r.v, mm);
    }
    return r;
}
// x == 0 (mod m) for x in [0, 2m): x is 0 or m
template <class F> H2V_HD bool fe_is_zero_lazy(const fe &x) {
    uint32_t z = 0, e = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        z |= x.v[i];
        e |= x.v[i] ^ F::m(i);
    }
    return z == 0 || e == 0;
}
// Cheap conditional -2m decided by the top limb alone: subtracts when x.v[7] > top(2m), so that (with T = top(2m),
// theta = (T+1) 2^224 > 2m) any x < theta + 2m comes out in [0, theta).  The NTT butterflies then keep every value
// below theta + 2m (< 2^256, and still small enough for fe_mul_lazy to return < 2m): a predicated 8-instruction
// subtraction instead of subtract + 8 selects.
template <class F> H2V_HD void fe_csub_2m_top(fe &t) {
    if (t.v[7] > fe_2m_limb<F>(7)) {
        uint32_t mm[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) mm[i] = fe_2m_limb<F>(i);
        uint32_t d[8];
        raw_sub(d, t.v, mm);
#pragma unroll
        for (int i = 0; i < 8; ++i) t.v[i] = d[i];
    }
}
// a + b and a + 2m - b without reduction
H2V_HD fe fe_add_raw(const fe &a, const fe &b) {
    fe r;
    raw_add(r.v, a.v, b.v);
    return r;
}
template <class F> H2V_HD fe fe_sub_plus_2m(const fe &a, const fe &b) {
    uint32_t mm[8];
    fe d, r;
#pragma unroll
    for (int i = 0; i < 8; ++i) mm[i] = fe_2m_limb<F>(i);
    raw_sub(d.v, mm, b.v);       // 2m - b > 0 for b < 2m
    raw_add(r.v, a.v, d.v);
    return r;
}
template <class F> H2V_HD fe fe_sqr(const fe &a) {
#ifdef __CUDA_ARCH__
    fe r = fe_sqr_lazy<F>(a);      // a canonical: the dedicated squaring (108 instead of 136 wide multiply-adds)
    fe_reduce_once<F>(r);
    return r;
#else
    return fe_mul<F>(a, a);
#endif
}

template <class F> H2V_HD fe fe_to_mont(const fe &canon) {
    fe r2;
#pragma unroll
    for (int i = 0; i < 8; ++i) r2.v[i] = F::r2(i);
    return fe_mul<F>(canon, r2);
}
template <class F> H2V_HD fe fe_from_mont(const fe &a) {
    fe one = fe_zero();
    one.v[0] = 1;
    return fe_mul<F>(a, one);
}
// a^e, e given as 8 little-endian 32-bit limbs
template <class F> H2V_HD fe fe_pow(const fe &a, const uint32_t *e, int nbits = 256) {
    fe acc = fe_one<F>();
    for (int i = nbits - 1; i >= 0; --i) {
        acc = fe_sqr<F>(acc);
        if ((e[i >> 5] >> (i & 31)) & 1) acc = fe_mul<F>(acc, a);
    }
    return acc;
}
// a^e scanning only the significant bits of a small exponent
template <class F> H2V_HD fe fe_pow_small(const fe &a, uint32_t e) {
    fe acc = fe_one<F>();
    int top = 31;
    while (top >= 0 && !((e >> top) & 1u)) --top;
    for (int i = top; i >= 0; --i) {
        acc = fe_sqr<F>(acc);
        if ((e >> i) & 1u) acc = fe_mul<F>(acc, a);
    }
    return acc;
}
template <class F> H2V_HD fe fe_pow_u64(const fe &a, uint64_t e) {
    uint32_t ee[8] = {(uint32_t)e, (uint32_t)(e >> 32), 0, 0, 0, 0, 0, 0};
    return fe_pow<F>(a, ee, 64);
}
// a^(m-2) (Fermat); a == 0 -> 0
template <class F> H2V_HD fe fe_inv(const fe &a) {
    uint32_t e[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) e[i] = F::m(i);
    e[0] -= 2;   // low limbs of p and r are >= 2
    return fe_pow<F>(a, e, 254);
}

// ------------------------------------------------------------------ fast inversion (binary extended Euclid)
// Latency matters where ONE inversion sits on the critical path (affine normalisation of an MSM result,
// the root of the batch-inversion tree): ~500 shift/subtract steps on the ALU pipe instead of the ~380
// dependent Montgomery products of Fermat's a^(m-2).  Works on the stored integer a = x R and converts:
// (xR)^-1 * R^3 * R^-1 = x^-1 R.   a == 0 -> 0.
H2V_HD void raw_shr1(uint32_t *a, uint32_t top) {      // a = (top:a) >> 1
#pragma unroll
    for (int i = 0; i < 7; ++i) a[i] = (a[i] >> 1) | (a[i + 1] << 31);
    a[7] = (a[7] >> 1) | (top << 31);
}
H2V_HD bool raw_is_one(const uint32_t *a) {
    uint32_t o = a[0] ^ 1u;
#pragma unroll
    for (int i = 1; i < 8; ++i) o |= a[i];
    return o == 0;
}
template <class F> H2V_HD void half_mod(uint32_t *x, const uint32_t *mm) {   // x = x / 2 mod m, x < m
    if (x[0] & 1u) {
        uint32_t t[8];
        raw_add(t, x, mm);            // x + m < 2^255: no carry out
#pragma unroll
        for (int i = 0; i < 8; ++i) x[i] = t[i];
    }
    raw_shr1(x, 0);
}
template <class F> H2V_HD fe fe_inv_fast(const fe &a) {
    if (fe_is_zero(a)) return a;
    uint32_t mm[8], u[8], v[8], x1[8], x2[8], t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        mm[i] = F::m(i);
        u[i] = a.v[i];
        v[i] = mm[i];
        x1[i] = 0;
        x2[i] = 0;
    }
    x1[0] = 1;
    while (!raw_is_one(u) && !raw_is_one(v)) {
        while (!(u[0] & 1u)) {
            raw_shr1(u, 0);
            half_mod<F>(x1, mm);
        }
        while (!(v[0] & 1u)) {
            raw_shr1(v, 0);
            half_mod<F>(x2, mm);
        }
        uint32_t bw = raw_sub(t, u, v);
        if (!bw) {                    // u >= v
#pragma unroll
            for (int i = 0; i < 8; ++i) u[i] = t[i];
            bw = raw_sub(t, x1, x2);
#pragma unroll
            for (int i = 0; i < 8; ++i) x1[i] = t[i];
            if (bw) {
                raw_add(t, x1, mm);
#pragma unroll
                for (int i = 0; i < 8; ++i) x1[i] = t[i];
            }
        } else {
            raw_sub(t, v, u);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = t[i];
            bw = raw_sub(t, x2, x1);
#pragma unroll
            for (int i = 0; i < 8; ++i) x2[i] = t[i];
            if (bw) {
                raw_add(t, x2, mm);
#pragma unroll
                for (int i = 0; i < 8; ++i) x2[i] = t[i];
            }
        }
    }
    fe r, r3;
    const bool uo = raw_is_one(u);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        r.v[i] = uo ? x1[i] : x2[i];
        r3.v[i] = F::r3(i);
    }
    return fe_mul<F>(r, r3);
}

}  // namespace h2v
