// zk_chips.hpp -- the reference's three chips, call by call (SURVEY.md 8(f) row 4, App. E).
//
//   FixedPointChip  /root/reference/src/gadget/fixed_point.rs      (each method cites its lines)
//   DistanceChip    /root/reference/src/gadget/distance.rs
//   VectorDBChip    /root/reference/src/gadget/vectordb.rs
// on top of the halo2-base primitives of zk_builder.hpp.  Same method names, argument order and failure behaviour
// (upstream panics <-> C++ exceptions, turned into H2V_EINVAL at the C ABI).
#pragma once
#include <functional>

#include "poseidon.hpp"
#include "zk_builder.hpp"

namespace h2v {
namespace zk {

// fixed_point.rs:42-215
struct FixedPointChip {
    RangeChip range;
    unsigned precision_bits, lookup_bits;
    U256 quantization_scale;      // 2^P
    U256 max_value;               // 2^(2P)
    U256 bn254_max;               // r - 1
    U256 negative_point;          // r - 2^(2P+1)
    std::vector<U256> pow_of_two;

    FixedPointChip(unsigned precision, unsigned lb) : range(lb), precision_bits(precision), lookup_bits(lb) {      // :54-98
        if (precision > 63) throw std::runtime_error("support only precision bits <= 63");
        if (precision < 32) throw std::runtime_error("support only precision bits >= 32");
        quantization_scale = u_pow2(precision);
        bn254_max = u_sub(f_modulus(), u_from(1));
        negative_point = f_add(f_sub(bn254_max, f_from_u(u_pow2(2 * precision + 1))), u_from(1));
        max_value = u_pow2(2 * precision);
        pow_of_two = range.gate.pow_of_two;
    }
    const GateChip &gate() const { return range.gate; }

    // :104-119
    U256 quantization(double x) const {
        const bool negative = signbit(x) && !isnan(x);      // f64::signum: -1.0 for every negative-signed value, -0.0 included
        const double scaled = round(fabs(x) * (double)((u128)1 << precision_bits));
        u128 xq;      // Rust `as u128` saturates
        if (!(scaled > 0)) xq = 0;
        else if (scaled >= 340282366920938463463374607431768211456.0) xq = ~(u128)0;
        else xq = (u128)scaled;
        U256 v = u_from128(xq);
        if (negative) v = f_add(f_sub(bn254_max, v), u_from(1));
        return v;
    }
    // :121-136
    double dequantization(const U256 &x) const {
        U256 m = x;
        double sign = 1.0;
        if (u_cmp(x, negative_point) > 0) {
            m = f_sub(f_sub(bn254_max, x), u_from(1));
            sign = -1.0;
        }
        const u128 lo = ((u128)m.l[1] << 64) | m.l[0];
        const u128 scale = (u128)1 << precision_bits;
        const double x_int = (double)(lo / scale);
        const double x_frac = (double)(lo % scale) / (double)scale;
        return sign * (x_int + x_frac);
    }
    std::vector<U256> quantize_vector(const std::vector<double> &v) const {      // fixed_point_vec.rs:30-32
        std::vector<U256> out;
        for (double x : v) out.push_back(quantization(x));
        return out;
    }
    std::vector<QCell> poly_constants(const double *c, size_t n) const {
        std::vector<QCell> out;
        for (size_t i = 0; i < n; ++i) out.push_back(Constant(quantization(c[i])));
        return out;
    }
    std::vector<QCell> generate_exp2_poly() const {      // :138-160
        static const double c[] = {3.6240421303547230336183979205877e-11, 4.1284327467833130245549169910389e-10,
                                   0.0000000071086385644026346316624185550542, 0.00000010172297085296590958930245291448,
                                   0.0000013215904023658396206789543841996, 0.000015252713316417140696221389106544,
                                   0.00015403531076657894204857389177279, 0.0013333558131297097698435464957392,
                                   0.0096181291078409107025643582456283, 0.055504108664804181586140094858174,
                                   0.24022650695910142332414229540187, 0.69314718055994529934452147700678, 1.0};
        return poly_constants(c, sizeof c / sizeof c[0]);
    }
    std::vector<QCell> generate_log_poly() const {      // :162-187
        static const double c[] = {-3.319586265362338e-08, 1.4957235315170112e-06, -3.1350053389526744e-05, 0.00040554177582512901,
                                   -0.0036218342998850703, 0.023663846121538389, -0.11691877183255484, 0.44524062371564499,
                                   -1.3195777548208449, 3.0518128028712077, -5.4904626000399528, 7.6298580090181591,
                                   -8.1653313719804235, 7.1389971101896279, -3.1937385492842112};
        return poly_constants(c, sizeof c / sizeof c[0]);
    }
    std::vector<QCell> generate_sin_poly() const {      // :189-214
        static const double c[] = {-1.1008071636607462e-11, 2.4208013888629323e-10, -3.8584805817996712e-10, -2.3786993104309845e-08,
                                   -2.9795813710683115e-09, 2.7608543130047009e-06, -6.4467066994122565e-09, -0.00019840680551418068,
                                   -3.839555844512214e-09, 0.0083333350601673614, -5.0943769725466814e-10, -0.16666666657583049,
                                   -8.5029878414113731e-12, 1.0000000000003146, -1.9323057584419828e-15};
        return poly_constants(c, sizeof c / sizeof c[0]);
    }

    Assigned qadd(Context &ctx, const QCell &a, const QCell &b) const { return gate().add(ctx, a, b); }      // :487-497
    Assigned qsub(Context &ctx, const QCell &a, const QCell &b) const { return gate().sub(ctx, a, b); }      // :499-509
    Assigned neg(Context &ctx, const QCell &a) const { return gate().neg(ctx, a); }                          // :294-299
    Assigned qsum(Context &ctx, const std::vector<QCell> &a) const { return gate().sum(ctx, a); }            // :287-292
    // :523-539
    Assigned is_neg(Context &ctx, const QCell &a) const {
        const auto dm = range.div_mod(ctx, a, u_pow2(2 * precision_bits + 1), 254);
        const Assigned is_pos = gate().is_zero(ctx, dm.first);
        return gate().not_(ctx, Existing(is_pos));
    }
    // :511-521
    Assigned qabs(Context &ctx, const QCell &a) const {
        const Assigned a_reverse = gate().neg(ctx, a);
        const Assigned n = is_neg(ctx, a);
        return gate().select(ctx, Existing(a_reverse), a, Existing(n));
    }
    // :541-556
    Assigned cond_neg(Context &ctx, const QCell &a, const Assigned &is_neg_) const {
        const Assigned neg_a = gate().neg(ctx, a);
        return gate().select(ctx, Existing(neg_a), a, Existing(is_neg_));
    }
    // :558-569
    Assigned sign(Context &ctx, const QCell &a) const {
        const Assigned neg_one = gate().neg(ctx, Constant(1));
        const Assigned n = is_neg(ctx, a);
        return gate().select(ctx, Existing(neg_one), Constant(1), Existing(n));
    }
    // :571-586
    Assigned clip(Context &ctx, const QCell &a) const {
        const Assigned s = is_neg(ctx, a);
        const Assigned a_abs = qabs(ctx, a);
        const auto dm = range.div_mod(ctx, Existing(a_abs), max_value, 254);
        return cond_neg(ctx, Existing(dm.second), s);
    }
    // :974-1016
    std::pair<Assigned, Assigned> signed_div_scale(Context &ctx, const QCell &a) const {
        const U256 b = quantization_scale;
        const bool a_is_neg = u_cmp(a.v, u_pow2(252)) > 0;
        U256 q, r;
        if (a_is_neg) {
            const U256 a_abs = f_add(f_sub(bn254_max, a.v), u_from(1));
            U256 dq, dr;
            u_divmod(a_abs, b, dq, dr);
            if (!u_is_zero(dr)) dq = u_add(dq, u_from(1));      // div_ceil
            q = u_add(u_sub(bn254_max, dq), u_from(1));           // r - ceil(|a| / b)
            r = u_sub(a.v, f_mul(f_from_u(b), f_from_u(q)));
        } else {
            u_divmod(a.v, b, q, r);
        }
        ctx.assign_region({Witness(f_from_u(r), OP_SDS_R, R(3), 0, 0, precision_bits), Constant(f_from_u(b)),
                           Witness(f_from_u(q), OP_SDS_Q, R(3), 0, 0, precision_bits), a},
                          {0});
        const Assigned rem = ctx.get(-4), div = ctx.get(-2);
        range.check_big_less_than_safe(ctx, rem, b);
        const Assigned div_abs = qabs(ctx, Existing(div));
        range.check_big_less_than_safe(ctx, div_abs, u_pow2(precision_bits * 3));
        return {div, rem};
    }
    // :588-604
    Assigned qmul(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned ab = gate().mul(ctx, a, b);
        return signed_div_scale(ctx, Existing(ab)).first;
    }
    // :797-815 (the impl's override of the trait default at :267-285; same body)
    Assigned bit_xor(Context &ctx, const QCell &a_, const QCell &b_) const {
        const Assigned a = gate().add(ctx, Constant(0), a_);
        const Assigned b = gate().add(ctx, Constant(0), b_);
        gate().assert_bit(ctx, a);
        gate().assert_bit(ctx, b);
        const Assigned ab = gate().add(ctx, Existing(a), Existing(b));
        const Assigned one = gate().add(ctx, Constant(1), Constant(0));
        return gate().is_equal(ctx, Existing(ab), Existing(one));
    }
    // :606-629
    Assigned qmod(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned a_sign = is_neg(ctx, a);
        const Assigned b_sign = is_neg(ctx, b);
        gate().assert_is_const(ctx, b_sign, u_zero());
        const Assigned a_abs = qabs(ctx, a);
        const auto dm = range.div_mod_var(ctx, Existing(a_abs), b, precision_bits * 4, precision_bits * 2);
        const Assigned res_abs_comp = gate().sub(ctx, b, Existing(dm.second));
        return gate().select(ctx, Existing(res_abs_comp), Existing(dm.second), Existing(a_sign));
    }
    // :631-656
    Assigned qdiv(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned a_sign = is_neg(ctx, a);
        const Assigned b_sign = is_neg(ctx, b);
        const Assigned a_abs = qabs(ctx, a);
        const Assigned b_abs = qabs(ctx, b);
        const Assigned a_rescale = gate().mul(ctx, Existing(a_abs), Constant(quantization_scale));
        const auto dm = range.div_mod_var(ctx, Existing(a_rescale), Existing(b_abs), precision_bits * 4, precision_bits * 2);
        const Assigned ab_sign = bit_xor(ctx, Existing(a_sign), Existing(b_sign));
        return cond_neg(ctx, Existing(dm.first), ab_sign);
    }
    // :658-686 (Horner, highest degree first)
    Assigned polynomial(Context &ctx, const QCell &x, const std::vector<QCell> &coef) const {
        QCell last_y = Constant(0);
        Assigned result = qadd(ctx, x, Constant(0));
        for (size_t idx = 0; idx < coef.size(); ++idx) {
            const Assigned y_add = qadd(ctx, last_y, coef[idx]);
            last_y = Existing(y_add);
            if (idx + 1 < coef.size()) {
                const Assigned y = qmul(ctx, x, Existing(y_add));
                last_y = Existing(y);
            } else {
                result = y_add;
            }
        }
        return result;
    }
    // :688-708
    void check_power_of_two(Context &ctx, const Assigned &pow2_exponent, const Assigned &exponent) const {
        const std::vector<Assigned> bits = gate().num_to_bits(ctx, pow2_exponent, precision_bits * 2);
        std::vector<QCell> qb;
        for (const Assigned &b : bits) qb.push_back(Existing(b));
        const Assigned sum_of_bits = gate().sum(ctx, qb);
        const Assigned sum_m1 = gate().sub(ctx, Existing(sum_of_bits), Constant(1));
        const Assigned z = gate().is_zero(ctx, sum_m1);
        gate().assert_is_const(ctx, z, u_from(1));
        const Assigned bit = gate().select_from_idx(ctx, qb, Existing(exponent));
        const Assigned bit_m1 = gate().sub(ctx, Existing(bit), Constant(1));
        const Assigned z2 = gate().is_zero(ctx, bit_m1);
        gate().assert_is_const(ctx, z2, u_from(1));
    }
    // :710-734
    Assigned qexp2(Context &ctx, const QCell &a) const {
        const Assigned a_abs = qabs(ctx, a);
        const auto dm = range.div_mod(ctx, Existing(a_abs), u_pow2(precision_bits), precision_bits * 2);
        std::vector<QCell> pows;
        for (const U256 &p : pow_of_two) pows.push_back(Constant(p));
        const Assigned int_part_pow2 = gate().select_from_idx(ctx, pows, Existing(dm.first));
        const Assigned y_frac = polynomial(ctx, Existing(dm.second), generate_exp2_poly());
        const Assigned res_pos = gate().mul(ctx, Existing(int_part_pow2), Existing(y_frac));
        const Assigned res_neg = qdiv(ctx, Constant(quantization_scale), Existing(res_pos));
        const Assigned n = is_neg(ctx, a);
        return gate().select(ctx, Existing(res_neg), Existing(res_pos), Existing(n));
    }
    // :736-795
    Assigned qlog2(Context &ctx, const QCell &a) const {
        const Assigned a_assigned = gate().add(ctx, a, Constant(0));
        const Assigned n = is_neg(ctx, a);
        const Assigned z = gate().is_zero(ctx, a_assigned);
        const Assigned is_invalid = gate().or_(ctx, Existing(n), Existing(z));
        gate().assert_is_const(ctx, is_invalid, u_zero());
        const unsigned num_bits = precision_bits * 2;
        uint64_t num_digits = 1;      // index of the highest set bit (1 when there is none, as the fold's seed)
        for (unsigned i = 0; i < 256; ++i)
            if (u_bit(a_assigned.v, i)) num_digits = i;
        if (num_digits >= gate().pow_of_two.size()) throw std::runtime_error("index out of bounds: pow_of_two");
        const U256 pow1 = gate().pow_of_two[num_digits];
        const Assigned pow1_witness = gate().add(ctx, Witness(pow1, OP_POW2_MSB, a_assigned.off), Constant(0));
        const Assigned exp1 = gate().add(ctx, Witness(u_from(num_digits), OP_MSB, a_assigned.off), Constant(0));
        check_power_of_two(ctx, pow1_witness, exp1);
        const Assigned pow2_witness = gate().mul(ctx, Existing(pow1_witness), Constant(2));
        const Assigned exp2 = gate().add(ctx, Existing(exp1), Constant(1));
        check_power_of_two(ctx, pow2_witness, exp2);
        const Assigned a_lt_pow2 = range.is_less_than(ctx, a, Existing(pow2_witness), num_bits);
        const Assigned a_gt_pow1 = range.is_less_than(ctx, Existing(pow1_witness), a, num_bits);
        const Assigned a_eq_pow1 = gate().is_equal(ctx, a, Existing(pow1_witness));
        const Assigned a_ge_pow1 = gate().or_(ctx, Existing(a_eq_pow1), Existing(a_gt_pow1));
        const Assigned a_bound = gate().and_(ctx, Existing(a_lt_pow2), Existing(a_ge_pow1));
        gate().assert_is_const(ctx, a_bound, u_from(1));
        // shift a into [2, 4)
        const Assigned shift = gate().sub(ctx, Constant(precision_bits + 2), Existing(exp2));
        const Assigned is_shift_neg = is_neg(ctx, Existing(shift));
        const Assigned shift_abs = qabs(ctx, Existing(shift));
        const uint64_t sidx = shift_abs.v.l[0] & 0xffffffffull;
        if (sidx >= gate().pow_of_two.size()) throw std::runtime_error("index out of bounds: pow_of_two");
        const Assigned shift_pow2_witness = gate().add(ctx, Witness(gate().pow_of_two[sidx], OP_POW2_LOW32, shift_abs.off), Constant(0));
        check_power_of_two(ctx, shift_pow2_witness, shift_abs);
        const Assigned a_ls = gate().mul(ctx, a, Existing(shift_pow2_witness));
        const auto dm = range.div_mod_var(ctx, a, Existing(shift_pow2_witness), num_bits, precision_bits + 1);
        const Assigned a_norm = gate().select(ctx, Existing(dm.first), Existing(a_ls), Existing(is_shift_neg));
        const Assigned log_a_norm = polynomial(ctx, Existing(a_norm), generate_log_poly());
        const Assigned log_shift = gate().neg(ctx, Existing(shift));
        const Assigned log_shift_q = gate().mul(ctx, Existing(log_shift), Constant(quantization_scale));
        return gate().add(ctx, Existing(log_a_norm), Existing(log_shift_q));
    }
    // :817-841
    Assigned qsin(Context &ctx, const QCell &a) const {
        const Assigned a_abs = qabs(ctx, a);
        const Assigned a_sign = is_neg(ctx, a);
        const QCell pi_2 = Constant(quantization(M_PI * 2.0));
        const Assigned a_mod = qmod(ctx, Existing(a_abs), pi_2);
        const QCell pi = Constant(quantization(M_PI));
        const Assigned a_mpi = qsub(ctx, Existing(a_mod), pi);
        const Assigned is_neg_a_mpi = is_neg(ctx, Existing(a_mpi));
        const Assigned sin_a_mod = polynomial(ctx, Existing(a_mod), generate_sin_poly());
        const Assigned sin_a_mpi_rev = polynomial(ctx, Existing(a_mpi), generate_sin_poly());
        const Assigned sin_a_mpi = neg(ctx, Existing(sin_a_mpi_rev));
        const Assigned sin_a_abs = gate().select(ctx, Existing(sin_a_mod), Existing(sin_a_mpi), Existing(is_neg_a_mpi));
        return cond_neg(ctx, Existing(sin_a_abs), a_sign);
    }
    // :843-852
    Assigned qcos(Context &ctx, const QCell &a) const {
        const Assigned half_pi = ctx.load_constant(quantization(M_PI_2));
        const Assigned s = qadd(ctx, a, Existing(half_pi));
        return qsin(ctx, Existing(s));
    }
    // :383-393
    Assigned qtan(Context &ctx, const QCell &a) const {
        const Assigned s = qsin(ctx, a);
        const Assigned c = qcos(ctx, a);
        return qdiv(ctx, Existing(s), Existing(c));
    }
    // :854-874
    Assigned inner_product(Context &ctx, const std::vector<QCell> &a, const std::vector<QCell> &b) const {
        if (a.size() != b.size()) throw std::runtime_error("assertion failed: a.len() == b.len()");
        Assigned res = qadd(ctx, Constant(0), Constant(0));
        for (size_t i = 0; i < a.size(); ++i) {
            const Assigned ab = qmul(ctx, a[i], b[i]);
            res = qadd(ctx, Existing(res), Existing(ab));
        }
        return res;
    }
    // :876-886
    Assigned qexp(Context &ctx, const QCell &a) const {
        const Assigned ln2 = ctx.load_constant(quantization(log(2.0)));
        const Assigned x1 = qdiv(ctx, a, Existing(ln2));
        return qexp2(ctx, Existing(x1));
    }
    // :954-964
    Assigned qlog(Context &ctx, const QCell &a) const {
        const Assigned log2e = ctx.load_constant(quantization(M_LOG2E));
        const Assigned log2a = qlog2(ctx, a);
        return qdiv(ctx, Existing(log2a), Existing(log2e));
    }
    // :441-456
    Assigned qpow(Context &ctx, const QCell &x, const QCell &exponent) const {
        const Assigned logx = qlog(ctx, x);
        const Assigned alogx = qmul(ctx, exponent, Existing(logx));
        return qexp(ctx, Existing(alogx));
    }
    // :966-972
    Assigned qsqrt(Context &ctx, const QCell &x) const {
        const Assigned half = ctx.load_constant(quantization(0.5));
        return qpow(ctx, x, Existing(half));
    }
    // :888-916
    Assigned qsinh_cosh(Context &ctx, const QCell &a, bool cosh_) const {
        const Assigned ea = qexp(ctx, a);
        const Assigned na = neg(ctx, a);
        const Assigned ena = qexp(ctx, Existing(na));
        const Assigned nume = cosh_ ? qadd(ctx, Existing(ea), Existing(ena)) : qsub(ctx, Existing(ea), Existing(ena));
        const Assigned two = ctx.load_constant(quantization(2.0));
        return qdiv(ctx, Existing(nume), Existing(two));
    }
    Assigned qsinh(Context &ctx, const QCell &a) const { return qsinh_cosh(ctx, a, false); }
    Assigned qcosh(Context &ctx, const QCell &a) const { return qsinh_cosh(ctx, a, true); }
    // :407-417
    Assigned qtanh(Context &ctx, const QCell &a) const {
        const Assigned s = qsinh(ctx, a);
        const Assigned c = qcosh(ctx, a);
        return qdiv(ctx, Existing(s), Existing(c));
    }
    // :918-934
    Assigned qmax(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned amb = qsub(ctx, a, b);
        const Assigned s = is_neg(ctx, Existing(amb));
        return gate().select(ctx, b, a, Existing(s));
    }
    // :936-952
    Assigned qmin(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned amb = qsub(ctx, a, b);
        const Assigned s = is_neg(ctx, Existing(amb));
        return gate().select(ctx, a, b, Existing(s));
    }
};

inline std::vector<QCell> existing(const std::vector<Assigned> &v) {
    std::vector<QCell> out;
    out.reserve(v.size());
    for (const Assigned &a : v) out.push_back(Existing(a));
    return out;
}

// distance.rs:15-195
struct DistanceChip {
    const FixedPointChip &fp;
    explicit DistanceChip(const FixedPointChip &f) : fp(f) {}
    // :97-119
    Assigned euclidean_distance(Context &ctx, const std::vector<Assigned> &a, const std::vector<Assigned> &b) const {
        if (a.size() != b.size()) throw std::runtime_error("assertion failed: a.len() == b.len()");
        std::vector<Assigned> ab;
        for (size_t i = 0; i < a.size(); ++i) ab.push_back(fp.qsub(ctx, Existing(a[i]), Existing(b[i])));
        const Assigned dist_square = fp.inner_product(ctx, existing(ab), existing(ab));
        return fp.qsqrt(ctx, Existing(dist_square));
    }
    // :121-144
    Assigned cosine_distance(Context &ctx, const std::vector<Assigned> &a, const std::vector<Assigned> &b) const {
        if (a.size() != b.size()) throw std::runtime_error("assertion failed: a.len() == b.len()");
        const Assigned ab = fp.inner_product(ctx, existing(a), existing(b));
        const Assigned aa = fp.inner_product(ctx, existing(a), existing(a));
        const Assigned bb = fp.inner_product(ctx, existing(b), existing(b));
        const Assigned aa_sqrt = fp.qsqrt(ctx, Existing(aa));
        const Assigned bb_sqrt = fp.qsqrt(ctx, Existing(bb));
        const Assigned denom = fp.qmul(ctx, Existing(aa_sqrt), Existing(bb_sqrt));
        const Assigned sim = fp.qdiv(ctx, Existing(ab), Existing(denom));
        const Assigned one = ctx.load_constant(fp.quantization(1.0));
        return fp.qsub(ctx, Existing(one), Existing(sim));
    }
    // :146-175 (the count and the length re-enter as unconstrained witnesses, as upstream)
    Assigned hamming_distance(Context &ctx, const std::vector<Assigned> &a, const std::vector<Assigned> &b) const {
        if (a.size() != b.size()) throw std::runtime_error("assertion failed: a.len() == b.len()");
        std::vector<Assigned> ab;
        for (size_t i = 0; i < a.size(); ++i) ab.push_back(fp.gate().is_equal(ctx, Existing(a[i]), Existing(b[i])));
        const Assigned ab_sum = fp.gate().sum(ctx, existing(ab));
        const Assigned len = ctx.load_witness(Witness(fp.quantization((double)a.size()), RULE_CONST, 0));
        const u128 lo = ((u128)ab_sum.v.l[1] << 64) | ab_sum.v.l[0];
        const Assigned ab_sum_q = ctx.load_witness(Witness(fp.quantization((double)lo), OP_QCOUNT, ab_sum.off, 0, 0, fp.precision_bits));
        const Assigned sim = fp.qdiv(ctx, Existing(ab_sum_q), Existing(len));
        const Assigned one = ctx.load_constant(fp.quantization(1.0));
        return fp.qsub(ctx, Existing(one), Existing(sim));
    }
    // :177-195
    Assigned manhattan_distance(Context &ctx, const std::vector<Assigned> &a, const std::vector<Assigned> &b) const {
        if (a.size() != b.size()) throw std::runtime_error("assertion failed: a.len() == b.len()");
        std::vector<Assigned> diff, abs_;
        for (size_t i = 0; i < a.size(); ++i) diff.push_back(fp.qsub(ctx, Existing(a[i]), Existing(b[i])));
        for (const Assigned &d : diff) abs_.push_back(fp.qabs(ctx, Existing(d)));
        return fp.gate().sum(ctx, existing(abs_));
    }
};

// halo2-base's `poseidon` crate (PoseidonChip<F, T, RATE>, adapted from Scroll / PSE `poseidon::Spec`) [UPSTREAM, recalled]:
// the optimised form -- pre-multiplied round constants, `pre_sparse_mds` and one sparse matrix per partial round --
// laid out as gate cells.  The factorisation is derived here (same algebra as poseidon.hpp's host sponge, arranged the
// way `Spec::calculate_*` arranges it) and the permutation result is checked against the plain round function, which the
// published Poseidon vectors pin (tests/test_circuit.py).
struct PoseidonChip3 {      // T = 3, RATE = 2 (examples/query.rs:27-30)
    static constexpr int T = 3, RATE = 2;
    int r_f, r_p;
    U256 mds[T][T], pre_sparse[T][T];
    std::vector<std::vector<U256>> start, end;      // r_f/2 and r_f/2 - 1 rows of T optimised constants
    std::vector<U256> partial;                      // r_p
    struct Sparse {
        U256 row[T], col_hat[T - 1];
    };
    std::vector<Sparse> sparse;
    Assigned init_state[T], state[T];
    std::vector<Assigned> absorbing;

    static void mat_mul(const U256 (&a)[T][T], const U256 (&b)[T][T], U256 (&o)[T][T]) {
        U256 t[T][T];
        for (int i = 0; i < T; ++i)
            for (int j = 0; j < T; ++j) {
                U256 acc = u_zero();
                for (int k = 0; k < T; ++k) acc = f_add(acc, f_mul(a[i][k], b[k][j]));
                t[i][j] = acc;
            }
        memcpy(o, t, sizeof t);
    }
    static void mat_vec(const U256 (&a)[T][T], const U256 *v, U256 *o) {
        U256 t[T];
        for (int i = 0; i < T; ++i) {
            U256 acc = u_zero();
            for (int k = 0; k < T; ++k) acc = f_add(acc, f_mul(a[i][k], v[k]));
            t[i] = acc;
        }
        for (int i = 0; i < T; ++i) o[i] = t[i];
    }
    template <int N> static void inverse(const U256 (&a)[N][N], U256 (&o)[N][N]) {
        Fr64 m[N][N], mi[N][N];
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j) m[i][j] = frh::to_mont(as_fr(a[i][j]));
        poseidon_detail::mat_inverse<N>(m, mi);
        for (int i = 0; i < N; ++i)
            for (int j = 0; j < N; ++j) o[i][j] = as_u(frh::from_mont(mi[i][j]));
    }
    static void transpose(const U256 (&a)[T][T], U256 (&o)[T][T]) {
        U256 t[T][T];
        for (int i = 0; i < T; ++i)
            for (int j = 0; j < T; ++j) t[j][i] = a[i][j];
        memcpy(o, t, sizeof t);
    }

    // PoseidonChip::new(ctx, r_f, r_p): the spec, and the initial state [2^64, 0, 0] loaded as constants
    PoseidonChip3(Context &ctx, int rf, int rp) : r_f(rf), r_p(rp) {
        const PoseidonSpec<T> sp = poseidon_make_spec<T>(rf, rp);
        std::vector<std::vector<U256>> c((size_t)(rf + rp), std::vector<U256>(T));
        for (int r = 0; r < rf + rp; ++r)
            for (int i = 0; i < T; ++i) c[r][i] = as_u(frh::from_mont(sp.rc[(size_t)r * T + i]));
        for (int i = 0; i < T; ++i)
            for (int j = 0; j < T; ++j) mds[i][j] = as_u(frh::from_mont(sp.mds[i][j]));
        U256 inv[T][T];
        inverse<T>(mds, inv);
        const int half = rf / 2;
        // constants of the first half: c0 as is, the others moved in front of the previous round's MDS
        start.assign((size_t)half, std::vector<U256>(T));
        start[0] = c[0];
        for (int r = 1; r < half; ++r) mat_vec(inv, c[r].data(), start[r].data());
        // partial rounds, from the last one backwards: only word 0 keeps a constant, the rest is pushed to the round before
        std::vector<U256> acc = c[(size_t)half + rp];
        partial.assign((size_t)rp, u_zero());
        for (int r = rp - 1; r >= 0; --r) {
            U256 tmp[T];
            mat_vec(inv, acc.data(), tmp);
            partial[r] = tmp[0];
            tmp[0] = u_zero();
            for (int i = 0; i < T; ++i) acc[i] = f_add(tmp[i], c[(size_t)half + r][i]);
        }
        start.push_back(std::vector<U256>(T));
        mat_vec(inv, acc.data(), start.back().data());
        end.assign((size_t)half - 1, std::vector<U256>(T));
        for (int r = 0; r + 1 < half; ++r) mat_vec(inv, c[(size_t)half + rp + 1 + r].data(), end[r].data());
        // sparse factorisation of the partial rounds' matrices, from the last partial round backwards (state as a column
        // vector): acc = S D with D = diag(1, D^) applied first -- D fixes word 0, so it commutes with the one-word S-box
        // and moves into the matrix of the round before (acc <- D M) -- and S = [[row], [col_hat | I]].  The shape makes
        // the factors unique: D^ = acc[1.., 1..], col_hat = acc[1.., 0], row = (acc[0, 0], acc[0, 1..] D^^-1).
        U256 accm[T][T];
        memcpy(accm, mds, sizeof mds);
        sparse.resize((size_t)rp);
        for (int r = 0; r < rp; ++r) {
            U256 dh[T - 1][T - 1], dhi[T - 1][T - 1];
            for (int i = 0; i < T - 1; ++i)
                for (int j = 0; j < T - 1; ++j) dh[i][j] = accm[i + 1][j + 1];
            inverse<T - 1>(dh, dhi);
            Sparse s;
            s.row[0] = accm[0][0];
            for (int j = 0; j < T - 1; ++j) {
                U256 a2 = u_zero();
                for (int i = 0; i < T - 1; ++i) a2 = f_add(a2, f_mul(accm[0][i + 1], dhi[i][j]));
                s.row[j + 1] = a2;
            }
            for (int i = 0; i < T - 1; ++i) s.col_hat[i] = accm[i + 1][0];
            U256 d[T][T];
            for (int i = 0; i < T; ++i)
                for (int j = 0; j < T; ++j) d[i][j] = (i == 0 || j == 0) ? u_from(i == j ? 1 : 0) : dh[i - 1][j - 1];
            mat_mul(d, mds, accm);
            sparse[(size_t)(rp - 1 - r)] = s;
        }
        memcpy(pre_sparse, accm, sizeof accm);
        init_state[0] = ctx.load_constant(u_pow2(64));
        for (int i = 1; i < T; ++i) init_state[i] = ctx.load_constant(u_zero());
        clear();
    }
    void clear() {
        for (int i = 0; i < T; ++i) state[i] = init_state[i];
        absorbing.clear();
    }
    void update(const std::vector<Assigned> &v) { absorbing.insert(absorbing.end(), v.begin(), v.end()); }

    static Assigned x_power5_with_constant(Context &ctx, const GateChip &g, const Assigned &x, const U256 &c) {
        const Assigned x2 = g.mul(ctx, Existing(x), Existing(x));
        const Assigned x4 = g.mul(ctx, Existing(x2), Existing(x2));
        return g.mul_add(ctx, Existing(x), Existing(x4), Constant(c));
    }
    void sbox_full(Context &ctx, const GateChip &g, const U256 *c) {
        for (int i = 0; i < T; ++i) state[i] = x_power5_with_constant(ctx, g, state[i], c[i]);
    }
    void sbox_part(Context &ctx, const GateChip &g, const U256 &c) { state[0] = x_power5_with_constant(ctx, g, state[0], c); }
    void absorb_with_pre_constants(Context &ctx, const GateChip &g, const std::vector<Assigned> &in, const U256 *pre) {
        if ((int)in.size() >= T) throw std::runtime_error("assertion failed: inputs.len() < T");
        const size_t offset = in.size() + 1;
        state[0] = g.add(ctx, Existing(state[0]), Constant(pre[0]));
        for (size_t i = 0; i < in.size(); ++i) state[i + 1] = g.sum(ctx, {Existing(state[i + 1]), Existing(in[i]), Constant(pre[i + 1])});
        for (size_t i = offset; i < (size_t)T; ++i)
            state[i] = g.add(ctx, Existing(state[i]), Constant(i == offset ? f_add(u_from(1), pre[i]) : pre[i]));
    }
    void apply_mds(Context &ctx, const GateChip &g, const U256 (&m)[T][T]) {
        Assigned res[T];
        std::vector<QCell> s = {Existing(state[0]), Existing(state[1]), Existing(state[2])};
        for (int i = 0; i < T; ++i) res[i] = g.inner_product(ctx, s, {Constant(m[i][0]), Constant(m[i][1]), Constant(m[i][2])});
        for (int i = 0; i < T; ++i) state[i] = res[i];
    }
    void apply_sparse_mds(Context &ctx, const GateChip &g, const Sparse &m) {
        Assigned res[T];
        res[0] = g.inner_product(ctx, {Existing(state[0]), Existing(state[1]), Existing(state[2])},
                                 {Constant(m.row[0]), Constant(m.row[1]), Constant(m.row[2])});
        for (int i = 1; i < T; ++i) res[i] = g.mul_add(ctx, Existing(state[0]), Constant(m.col_hat[i - 1]), Existing(state[i]));
        for (int i = 0; i < T; ++i) state[i] = res[i];
    }
    void permutation(Context &ctx, const GateChip &g, const std::vector<Assigned> &inputs) {
        const int half = r_f / 2;
        absorb_with_pre_constants(ctx, g, inputs, start[0].data());
        for (int r = 1; r < half; ++r) {
            sbox_full(ctx, g, start[(size_t)r].data());
            apply_mds(ctx, g, mds);
        }
        sbox_full(ctx, g, start[(size_t)half].data());
        apply_mds(ctx, g, pre_sparse);
        for (int r = 0; r < r_p; ++r) {
            sbox_part(ctx, g, partial[(size_t)r]);
            apply_sparse_mds(ctx, g, sparse[(size_t)r]);
        }
        for (size_t r = 0; r < end.size(); ++r) {
            sbox_full(ctx, g, end[r].data());
            apply_mds(ctx, g, mds);
        }
        const U256 zeros[T] = {u_zero(), u_zero(), u_zero()};
        sbox_full(ctx, g, zeros);
        apply_mds(ctx, g, mds);
    }
    Assigned squeeze(Context &ctx, const GateChip &g) {
        std::vector<Assigned> in;
        in.swap(absorbing);
        const bool exact = in.size() % RATE == 0;
        for (size_t i = 0; i < in.size(); i += RATE) {
            std::vector<Assigned> chunk(in.begin() + (long)i, in.begin() + (long)std::min(in.size(), i + RATE));
            permutation(ctx, g, chunk);
        }
        if (exact) permutation(ctx, g, {});
        return state[1];
    }
};

typedef std::function<Assigned(Context &, const std::vector<Assigned> &, const std::vector<Assigned> &)> DistanceFn;

// vectordb.rs:15-362
struct VectorDBChip {
    const FixedPointChip &fp;
    explicit VectorDBChip(const FixedPointChip &f) : fp(f) {}
    // :122-163
    std::pair<std::vector<Assigned>, std::vector<Assigned>> nearest_vector(Context &ctx, const std::vector<Assigned> &query,
                                                                           const std::vector<std::vector<Assigned>> &vectors,
                                                                           const DistanceFn &distance) const {
        if (vectors.empty()) throw std::runtime_error("called `Option::unwrap()` on a `None` value");
        std::vector<Assigned> distances;
        for (const auto &v : vectors) distances.push_back(distance(ctx, v, query));
        Assigned min = distances[0];
        for (size_t i = 1; i < distances.size(); ++i) min = fp.qmin(ctx, Existing(min), Existing(distances[i]));
        std::vector<Assigned> ind;
        for (const Assigned &d : distances) ind.push_back(fp.gate().is_equal(ctx, Existing(min), Existing(d)));
        std::vector<Assigned> result;
        for (size_t i = 0; i < vectors[0].size(); ++i) {
            std::vector<QCell> col;
            for (const auto &v : vectors) col.push_back(Existing(v[i]));
            result.push_back(fp.gate().select_by_indicator(ctx, col, ind));
        }
        return {ind, result};
    }
    // :165-223
    Assigned merkle_commitment(Context &ctx, PoseidonChip3 &poseidon, const std::vector<std::vector<Assigned>> &vectors) const {
        std::vector<Assigned> leaves;
        for (const auto &v : vectors) {
            poseidon.clear();
            poseidon.update(v);
            leaves.push_back(poseidon.squeeze(ctx, fp.gate()));
        }
        const size_t num_hashes = leaves.size();
        if (num_hashes == 0) throw std::runtime_error("attempt to subtract with overflow");
        size_t num_leaves = 1;
        while (num_leaves < num_hashes) num_leaves <<= 1;
        if (num_leaves > num_hashes) {
            const Assigned z = ctx.load_zero();
            leaves.resize(num_leaves, z);
        }
        while (leaves.size() > 1) {
            std::vector<Assigned> next;
            for (size_t i = 0; i < leaves.size(); i += 2) {
                poseidon.clear();
                poseidon.update({leaves[i], leaves[i + 1]});
                next.push_back(poseidon.squeeze(ctx, fp.gate()));
            }
            leaves.swap(next);
        }
        return leaves[0];
    }
    // :225-362
    std::pair<std::vector<std::vector<Assigned>>, std::vector<std::vector<Assigned>>> kmeans(
        Context &ctx, const std::vector<std::vector<Assigned>> &vectors, size_t K, size_t I, const DistanceFn &distance) const {
        if (!(K < vectors.size())) throw std::runtime_error("assertion failed: K < vectors.len()");
        const Assigned one = ctx.load_constant(fp.quantization(1.0));
        const Assigned zero = ctx.load_zero();
        std::vector<std::vector<Assigned>> centroids(vectors.begin(), vectors.begin() + (long)K);
        std::vector<std::vector<Assigned>> cluster_indicators;
        for (size_t iter = 0; iter < I; ++iter) {
            cluster_indicators.clear();
            for (const auto &v : vectors) {
                std::vector<Assigned> distances;
                for (const auto &c : centroids) distances.push_back(distance(ctx, c, v));
                Assigned min = distances[0];
                for (size_t i = 1; i < K; ++i) min = fp.qmin(ctx, Existing(min), Existing(distances[i]));
                std::vector<Assigned> ind;
                for (const Assigned &d : distances) {
                    const Assigned eq = fp.gate().is_equal(ctx, Existing(min), Existing(d));
                    ind.push_back(fp.gate().select(ctx, Existing(one), Existing(zero), Existing(eq)));
                }
                cluster_indicators.push_back(ind);
            }
            std::vector<Assigned> cluster_sizes = cluster_indicators[0];
            for (size_t v = 1; v < cluster_indicators.size(); ++v)
                for (size_t c = 0; c < K; ++c) cluster_sizes[c] = fp.qadd(ctx, Existing(cluster_sizes[c]), Existing(cluster_indicators[v][c]));
            for (size_t cid = 0; cid < K; ++cid) {
                std::vector<std::vector<Assigned>> filtered;
                for (size_t v = 0; v < vectors.size(); ++v) {
                    const Assigned is_zero = fp.gate().is_zero(ctx, cluster_indicators[v][cid]);
                    std::vector<Assigned> f;
                    for (const Assigned &x : vectors[v]) f.push_back(fp.gate().select(ctx, Existing(zero), Existing(x), Existing(is_zero)));
                    filtered.push_back(f);
                }
                std::vector<Assigned> sum = filtered[0];
                for (size_t v = 1; v < filtered.size(); ++v)
                    for (size_t d = 0; d < sum.size(); ++d) sum[d] = fp.qadd(ctx, Existing(filtered[v][d]), Existing(sum[d]));
                std::vector<Assigned> mean;
                for (const Assigned &s : sum) mean.push_back(fp.qdiv(ctx, Existing(s), Existing(cluster_sizes[cid])));
                centroids[cid] = mean;
            }
        }
        return {centroids, cluster_indicators};
    }
};

}  // namespace zk
}  // namespace h2v
