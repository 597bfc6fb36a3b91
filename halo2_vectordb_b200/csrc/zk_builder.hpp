// zk_builder.hpp -- the step BEFORE the hot path (SURVEY.md 8(f) row 4): the execution trace of the reference's chips.
//
// Host-side restatement of what produces the advice / lookup columns the commit path consumes:
//   * halo2-base (axiom-crypto/halo2-lib, branch community-edition = v0.3.0, /root/reference/Cargo.toml:22) [UPSTREAM,
//     un-vendored]: `Context` (one execution thread, `builder.main(0)` at /root/reference/src/scaffold/mod.rs:61),
//     `GateChip` (the vertical gate q * (a + b c - d) on four consecutive cells) and `RangeChip` (limb decomposition +
//     lookup cells).  The cell layouts of every primitive are RECALLED from that crate (DESIGN.md 9 lists them); what
//     can be checked here is checked: every gate, lookup and copy constraint of the trace holds (tests/test_circuit.py,
//     the MockProver of scaffold mod.rs:265), and the chip results match the f64 computations of the reference's tests.
//   * the reference's own chips, which ARE in /root/reference and are followed call by call:
//     FixedPointChip (src/gadget/fixed_point.rs), DistanceChip (src/gadget/distance.rs), VectorDBChip
//     (src/gadget/vectordb.rs).
// Like upstream this is serial host code (a Context is single-threaded).  A recording Context also keeps one `Rule` per
// cell -- how the cell's value follows from the inputs and earlier cells -- so that witness.cu can replay the trace for
// many inputs on the GPU (halo2-base's `witness_gen_only` idea); a normal Context records nothing.
// Values are kept as canonical 256-bit integers (most of the work is bit / limb decomposition and integer division);
// the layouter (circuit.cu) converts to the Montgomery form of the C ABI.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "fr_host.hpp"

namespace h2v {
namespace zk {

// ------------------------------------------------------------------------------------------- 256-bit integers
struct U256 {
    uint64_t l[4];
    bool operator==(const U256 &o) const { return l[0] == o.l[0] && l[1] == o.l[1] && l[2] == o.l[2] && l[3] == o.l[3]; }
    bool operator!=(const U256 &o) const { return !(*this == o); }
};
struct U256Hash {
    size_t operator()(const U256 &a) const {
        uint64_t h = a.l[0] * 0x9e3779b97f4a7c15ull;
        h ^= (a.l[1] + 0x7f4a7c15ull) * 0xbf58476d1ce4e5b9ull;
        h ^= (a.l[2] + 0x1ce4e5b9ull) * 0x94d049bb133111ebull;
        h ^= (a.l[3] + 0x133111ebull) * 0xd6e8feb86659fd93ull;
        return (size_t)(h ^ (h >> 29));
    }
};
typedef unsigned __int128 u128;
inline U256 u_zero() { return U256{{0, 0, 0, 0}}; }
inline U256 u_from(uint64_t x) { return U256{{x, 0, 0, 0}}; }
inline U256 u_from128(u128 x) { return U256{{(uint64_t)x, (uint64_t)(x >> 64), 0, 0}}; }
inline bool u_is_zero(const U256 &a) { return (a.l[0] | a.l[1] | a.l[2] | a.l[3]) == 0; }
inline int u_cmp(const U256 &a, const U256 &b) {
    for (int i = 3; i >= 0; --i)
        if (a.l[i] != b.l[i]) return a.l[i] < b.l[i] ? -1 : 1;
    return 0;
}
inline U256 u_add(const U256 &a, const U256 &b) {      // wrapping
    U256 r;
    u128 c = 0;
    for (int i = 0; i < 4; ++i) {
        c += (u128)a.l[i] + b.l[i];
        r.l[i] = (uint64_t)c;
        c >>= 64;
    }
    return r;
}
inline U256 u_sub(const U256 &a, const U256 &b) {      // wrapping
    U256 r;
    u128 bw = 0;
    for (int i = 0; i < 4; ++i) {
        u128 d = (u128)a.l[i] - b.l[i] - (uint64_t)bw;
        r.l[i] = (uint64_t)d;
        bw = (d >> 64) & 1;
    }
    return r;
}
inline bool u_bit(const U256 &a, unsigned i) { return i < 256 && ((a.l[i >> 6] >> (i & 63)) & 1); }
inline int u_bits(const U256 &a) {      // BigUint::bits(): position of the highest set bit + 1
    for (int i = 3; i >= 0; --i)
        if (a.l[i]) return 64 * i + 64 - __builtin_clzll(a.l[i]);
    return 0;
}
inline U256 u_shl(const U256 &a, unsigned s) {
    U256 r = u_zero();
    if (s >= 256) return r;
    const unsigned w = s >> 6, b = s & 63;
    for (int i = 3; i >= (int)w; --i) {
        r.l[i] = a.l[i - w] << b;
        if (b && i - (int)w - 1 >= 0) r.l[i] |= a.l[i - w - 1] >> (64 - b);
    }
    return r;
}
inline U256 u_shr(const U256 &a, unsigned s) {
    U256 r = u_zero();
    if (s >= 256) return r;
    const unsigned w = s >> 6, b = s & 63;
    for (unsigned i = 0; i + w < 4; ++i) {
        r.l[i] = a.l[i + w] >> b;
        if (b && i + w + 1 < 4) r.l[i] |= a.l[i + w + 1] << (64 - b);
    }
    return r;
}
inline U256 u_pow2(unsigned e) { return u_shl(u_from(1), e); }
inline U256 u_low_bits(const U256 &a, unsigned nbits) {      // a mod 2^nbits
    if (nbits >= 256) return a;
    return u_sub(a, u_shl(u_shr(a, nbits), nbits));
}
// floor division (num-integer `div_mod_floor` on BigUint); the divisor must not be zero
inline void u_divmod(const U256 &a, const U256 &b, U256 &q, U256 &r) {
    if (u_is_zero(b)) throw std::runtime_error("attempt to divide by zero");      // BigUint division panics upstream
    q = u_zero();
    r = u_zero();
    for (int i = u_bits(a) - 1; i >= 0; --i) {
        r = u_shl(r, 1);
        if (u_bit(a, (unsigned)i)) r.l[0] |= 1;
        if (u_cmp(r, b) >= 0) {
            r = u_sub(r, b);
            q.l[i >> 6] |= 1ull << (i & 63);
        }
    }
}

// ------------------------------------------------------------------------------------------- Fr on canonical values
inline const U256 &f_modulus() {
    static const U256 m = {{frh::MOD[0], frh::MOD[1], frh::MOD[2], frh::MOD[3]}};
    return m;
}
inline Fr64 as_fr(const U256 &a) { return Fr64{{a.l[0], a.l[1], a.l[2], a.l[3]}}; }
inline U256 as_u(const Fr64 &a) { return U256{{a.l[0], a.l[1], a.l[2], a.l[3]}}; }
inline U256 f_add(const U256 &a, const U256 &b) { return as_u(frh::add(as_fr(a), as_fr(b))); }
inline U256 f_sub(const U256 &a, const U256 &b) { return as_u(frh::sub(as_fr(a), as_fr(b))); }
inline U256 f_neg(const U256 &a) { return as_u(frh::neg(as_fr(a))); }
inline U256 f_mul(const U256 &a, const U256 &b) { return as_u(frh::mul(frh::mul(as_fr(a), as_fr(b)), frh::R2)); }      // (ab/R) R^2 / R
inline U256 f_inv(const U256 &a) { return as_u(frh::from_mont(frh::inv(frh::to_mont(as_fr(a))))); }
inline U256 f_from_u(const U256 &a) {      // biguint_to_fe: reduce mod r (inputs here are below 2r)
    return u_cmp(a, f_modulus()) >= 0 ? u_sub(a, f_modulus()) : a;
}

// ------------------------------------------------------------------------------------------- Context
// How a cell's value is computed (recording builders only).  Operands a, b, c are trace offsets; a negative operand
// -1 - i names cell i of the region being assigned (it may come later in the trace than the cell it feeds).
enum RuleKind : uint8_t {
    RULE_NONE,                     // no rule: a recording with such a cell cannot become a program
    RULE_INPUT,                    // imm-th value passed to h2v_builder_assign_witnesses
    RULE_CONST,                    // the recorded value (constants, fixed witnesses)
    RULE_COPY,                     // the value of cell a
    OP_ADD, OP_SUB, OP_NEG, OP_MUL,
    OP_MUL_ADD,                    // a b + c
    OP_OR,                         // a + b - a b
    OP_IS_ZERO, OP_INV_OR_ONE,     // a == 0; a^-1, or 1 when a == 0
    OP_BITS,                       // (a >> (imm & 255)) mod 2^(imm >> 8), on the canonical integer
    OP_DIV_Q, OP_DIV_R,            // floor(a / b), a mod b (b == 0: "attempt to divide by zero")
    OP_SDS_Q, OP_SDS_R,            // signed_div_scale's q and r for the scale 2^imm
    OP_IND, OP_IND_VAL,            // idx_to_indicator: low32(a) == imm ? 1 : 0, and ? a : 0
    OP_SELECT_IND,                 // b != 0 ? a : c
    OP_MSB,                        // qlog2: index of the highest set bit of a (1 when a == 0)
    OP_POW2_MSB, OP_POW2_LOW32,    // 2^msb(a), 2^low32(a) (>= 254: "index out of bounds: pow_of_two")
    OP_QCOUNT,                     // quantization((double)low128(a)) at precision imm
    RULE_KINDS
};
struct Rule {
    int64_t a, b, c;
    uint32_t imm;
    uint8_t kind;
};
inline constexpr int64_t R(int i) { return -1 - (int64_t)i; }      // operand: cell i of the current region

// halo2-base `AssignedValue`: a value and the position of its cell in the execution trace
struct Assigned {
    U256 v;
    int64_t off;
};
// halo2-base `QuantumCell`
struct QCell {
    enum Kind : uint8_t { W, C, E } kind;
    U256 v;
    int64_t off;
    Rule rule;      // of a W cell; kept by recording builders only
};
inline QCell Witness(const U256 &v) { return QCell{QCell::W, v, -1, Rule{0, 0, 0, 0, RULE_NONE}}; }
// a witness cell and its rule (every Witness site of the chips)
inline QCell Witness(const U256 &v, RuleKind k, int64_t a, int64_t b = 0, int64_t c = 0, uint32_t imm = 0) {
    return QCell{QCell::W, v, -1, Rule{a, b, c, imm, k}};
}
inline QCell Constant(const U256 &v) { return QCell{QCell::C, v, -1, Rule{}}; }
inline QCell Constant(uint64_t v) { return QCell{QCell::C, u_from(v), -1, Rule{}}; }
inline QCell Existing(const Assigned &a) { return QCell{QCell::E, a.v, a.off, Rule{}}; }

// halo2-base `Context<F>` (src/lib.rs of that crate): the trace of one thread.  witness_gen_only = false, i.e. the
// keygen / mock form that also records selectors and copy constraints (CircuitBuilderStage::{Mock, Keygen});
// the prover stage replays the same cells with the pinned break points, so one form serves both.
struct Context {
    std::vector<U256> advice;
    std::vector<uint8_t> selector;
    std::vector<int64_t> cells_to_lookup;
    std::vector<std::pair<int64_t, int64_t>> advice_eq;         // advice_equality_constraints
    std::vector<std::pair<U256, int64_t>> constant_eq;          // constant_equality_constraints
    bool has_zero = false;
    Assigned zero_cell{};
    bool recording = false;
    std::vector<Rule> rules;      // one per cell when recording

    Assigned get(int64_t i) const {      // negative offsets count from the end, as upstream's `ctx.get`
        const int64_t o = i < 0 ? (int64_t)advice.size() + i : i;
        if (o < 0 || o >= (int64_t)advice.size()) throw std::runtime_error("Context::get out of range");
        return Assigned{advice[(size_t)o], o};
    }
    Assigned last() const { return get(-1); }
    // row: the first cell of the region q belongs to (operands R(i) of its rule are relative to it)
    void assign_cell(const QCell &q, int64_t row = -1) {
        advice.push_back(q.v);
        const int64_t here = (int64_t)advice.size() - 1;
        if (q.kind == QCell::C) constant_eq.emplace_back(q.v, here);
        else if (q.kind == QCell::E) advice_eq.emplace_back(here, q.off);
        if (recording) record(q, row < 0 ? here : row);
    }
    void record(const QCell &q, int64_t row) {
        Rule r{0, 0, 0, 0, RULE_CONST};
        if (q.kind == QCell::E) r = Rule{q.off, 0, 0, 0, RULE_COPY};
        else if (q.kind == QCell::W) {
            r = q.rule;
            for (int64_t *o : {&r.a, &r.b, &r.c})
                if (*o < 0) *o = row - 1 - *o;
        }
        rules.push_back(r);
    }
    void assign_region(std::initializer_list<QCell> cells, std::initializer_list<int> gates) {
        const size_t row = advice.size();
        for (const QCell &q : cells) assign_cell(q, (int64_t)row);
        selector.resize(advice.size(), 0);
        for (int g : gates) selector[row + (size_t)g] = 1;
    }
    void assign_region(const std::vector<QCell> &cells, const std::vector<int> &gates) {
        const size_t row = advice.size();
        for (const QCell &q : cells) assign_cell(q, (int64_t)row);
        selector.resize(advice.size(), 0);
        for (int g : gates) selector[row + (size_t)g] = 1;
    }
    // `assign_region_smart`: extra equalities between cells of the region (relative offsets)
    void assign_region_smart(std::initializer_list<QCell> cells, std::initializer_list<int> gates,
                             std::initializer_list<std::pair<int, int>> eqs) {
        const int64_t row = (int64_t)advice.size();
        assign_region(cells, gates);
        for (auto &e : eqs) advice_eq.emplace_back(row + e.first, row + e.second);
    }
    void constrain_equal(const Assigned &a, const Assigned &b) { advice_eq.emplace_back(a.off, b.off); }
    Assigned load_witness(const QCell &w) {
        assign_cell(w);
        selector.resize(advice.size(), 0);
        return last();
    }
    Assigned load_constant(const U256 &v) {
        assign_cell(Constant(v));
        selector.resize(advice.size(), 0);
        return last();
    }
    Assigned load_zero() {      // cached, as upstream
        if (!has_zero) {
            zero_cell = load_constant(u_zero());
            has_zero = true;
        }
        return zero_cell;
    }
};

// ------------------------------------------------------------------------------------------- GateChip
// halo2-base gates/flex_gate.rs `GateInstructions for GateChip` (GateStrategy::Vertical) [UPSTREAM, recalled]
struct GateChip {
    std::vector<U256> pow_of_two;      // 2^i, i < Fr::NUM_BITS = 254
    GateChip() {
        pow_of_two.reserve(254);
        for (unsigned i = 0; i < 254; ++i) pow_of_two.push_back(f_from_u(u_pow2(i)));
    }
    // | a | b | 1 | a + b |
    Assigned add(Context &ctx, const QCell &a, const QCell &b) const {
        ctx.assign_region({a, b, Constant(1), Witness(f_add(a.v, b.v), OP_ADD, R(0), R(1))}, {0});
        return ctx.last();
    }
    // | a - b | b | 1 | a |
    Assigned sub(Context &ctx, const QCell &a, const QCell &b) const {
        ctx.assign_region({Witness(f_sub(a.v, b.v), OP_SUB, R(3), R(1)), b, Constant(1), a}, {0});
        return ctx.get(-4);
    }
    // | a | -a | 1 | 0 |
    Assigned neg(Context &ctx, const QCell &a) const {
        ctx.assign_region({a, Witness(f_neg(a.v), OP_NEG, R(0)), Constant(1), Constant(0)}, {0});
        return ctx.get(-3);
    }
    // | 0 | a | b | a b |
    Assigned mul(Context &ctx, const QCell &a, const QCell &b) const {
        ctx.assign_region({Constant(0), a, b, Witness(f_mul(a.v, b.v), OP_MUL, R(1), R(2))}, {0});
        return ctx.last();
    }
    // | c | a | b | a b + c |
    Assigned mul_add(Context &ctx, const QCell &a, const QCell &b, const QCell &c) const {
        ctx.assign_region({c, a, b, Witness(f_add(f_mul(a.v, b.v), c.v), OP_MUL_ADD, R(1), R(2), R(0))}, {0});
        return ctx.last();
    }
    // | 0 | x | x | x |
    void assert_bit(Context &ctx, const Assigned &x) const {
        ctx.assign_region({Constant(0), Existing(x), Existing(x), Existing(x)}, {0});
    }
    void assert_is_const(Context &ctx, const Assigned &a, const U256 &c) const { ctx.constant_eq.emplace_back(c, a.off); }
    Assigned not_(Context &ctx, const QCell &a) const { return sub(ctx, Constant(1), a); }
    Assigned and_(Context &ctx, const QCell &a, const QCell &b) const { return mul(ctx, a, b); }
    // | 1 - b | 1 | b | 1 | b | a | 1 - b | a + b - a b |
    Assigned or_(Context &ctx, const QCell &a, const QCell &b) const {
        const U256 not_b = f_sub(u_from(1), b.v);
        const U256 out = f_sub(f_add(a.v, b.v), f_mul(a.v, b.v));
        ctx.assign_region_smart({Witness(not_b, OP_SUB, R(1), R(2)), Constant(1), b, Constant(1), b, a, Witness(not_b, OP_SUB, R(1), R(2)),
                                 Witness(out, OP_OR, R(5), R(2))},
                                {0, 4}, {{0, 6}, {2, 4}});
        return ctx.last();
    }
    // | a - b | 1 | b | a | b | sel | a - b | out |
    Assigned select(Context &ctx, const QCell &a, const QCell &b, const QCell &sel) const {
        const U256 diff = f_sub(a.v, b.v);
        const U256 out = f_add(f_mul(diff, sel.v), b.v);
        ctx.assign_region_smart({Witness(diff, OP_SUB, R(3), R(2)), Constant(1), b, a, b, sel, Witness(diff, OP_SUB, R(3), R(2)),
                                 Witness(out, OP_MUL_ADD, R(0), R(5), R(2))},
                                {0, 4}, {{0, 6}, {2, 4}});
        return ctx.last();
    }
    // | is_zero | a | inv | 1 | 0 | a | is_zero | 0 |
    Assigned is_zero(Context &ctx, const Assigned &a) const {
        const bool z = u_is_zero(a.v);
        const U256 isz = u_from(z ? 1 : 0), inv = z ? u_from(1) : f_inv(a.v);
        ctx.assign_region_smart({Witness(isz, OP_IS_ZERO, R(1)), Existing(a), Witness(inv, OP_INV_OR_ONE, R(1)), Constant(1), Constant(0),
                                 Existing(a), Witness(isz, OP_IS_ZERO, R(1)), Constant(0)},
                                {0, 4}, {{0, 6}, {1, 5}});
        return ctx.get(-2);
    }
    Assigned is_equal(Context &ctx, const QCell &a, const QCell &b) const {
        const Assigned diff = sub(ctx, a, b);
        return is_zero(ctx, diff);
    }
    // sum: | a0 | a1 | 1 | a0 + a1 | a2 | 1 | ... |
    Assigned sum(Context &ctx, const std::vector<QCell> &a) const {
        if (a.empty()) return ctx.load_zero();
        if (a.size() == 1) {
            ctx.assign_region({a[0]}, {});
            return ctx.last();
        }
        std::vector<QCell> cells;
        std::vector<int> gates;
        cells.reserve(1 + 3 * (a.size() - 1));
        U256 s = a[0].v;
        cells.push_back(a[0]);
        for (size_t i = 1; i < a.size(); ++i) {
            s = f_add(s, a[i].v);
            cells.push_back(a[i]);
            cells.push_back(Constant(1));
            cells.push_back(Witness(s, OP_ADD, R((int)(3 * i - 3)), R((int)(3 * i - 2))));
            gates.push_back((int)(3 * (i - 1)));
        }
        ctx.assign_region(cells, gates);
        return ctx.last();
    }
    // inner product: | 0 | a0 | b0 | s0 | a1 | b1 | s1 | ...; when b0 is the constant 1 the region starts at | a0 | a1 | b1 | ...
    Assigned inner_product(Context &ctx, const std::vector<QCell> &a, const std::vector<QCell> &b) const {
        if (a.size() != b.size() || a.empty()) throw std::runtime_error("inner_product: length mismatch");
        const bool starts_with_one = b[0].kind == QCell::C && b[0].v == u_from(1);
        std::vector<QCell> cells;
        std::vector<int> gates;
        U256 s;
        size_t first;
        if (starts_with_one) {
            s = a[0].v;
            cells.push_back(a[0]);
            first = 1;
        } else {
            s = u_zero();
            cells.push_back(Constant(0));
            first = 0;
        }
        for (size_t i = first; i < a.size(); ++i) {
            s = f_add(s, f_mul(a[i].v, b[i].v));
            const int prev = (int)cells.size() - 1;
            gates.push_back(prev);
            cells.push_back(a[i]);
            cells.push_back(b[i]);
            cells.push_back(Witness(s, OP_MUL_ADD, R(prev + 1), R(prev + 2), R(prev)));
        }
        ctx.assign_region(cells, gates);
        return ctx.last();
    }
    // little-endian bits of a, constrained by sum b_i 2^i = a and b_i (b_i - 1) = 0
    std::vector<Assigned> num_to_bits(Context &ctx, const Assigned &a, unsigned range_bits) const {
        std::vector<QCell> bits, pows;
        for (unsigned i = 0; i < range_bits; ++i) {
            bits.push_back(Witness(u_from(u_bit(a.v, i) ? 1 : 0), OP_BITS, a.off, 0, 0, i | 1u << 8));
            pows.push_back(Constant(pow_of_two[i]));
        }
        const int64_t row = (int64_t)ctx.advice.size();
        const Assigned acc = inner_product(ctx, bits, pows);
        ctx.constrain_equal(a, acc);
        std::vector<Assigned> cells;
        cells.push_back(ctx.get(row));
        for (unsigned i = 1; i < range_bits; ++i) cells.push_back(ctx.get(row + 1 + 3 * (int64_t)(i - 1)));
        for (const Assigned &b : cells) assert_bit(ctx, b);
        return cells;
    }
    // ind[i] (idx - i) = 0 and ind[i] boolean: | 0 | ind | idx | ind idx | -i | ind | 0 |, then assert_bit
    std::vector<Assigned> idx_to_indicator(Context &ctx, QCell idx, size_t len) const {
        std::vector<Assigned> ind;
        ind.reserve(len);
        const uint64_t idx_val = idx.v.l[0] & 0xffffffffull;      // get_lower_32
        for (size_t i = 0; i < len; ++i) {
            const bool hit = idx_val == i;
            const U256 ind_val = u_from(hit ? 1 : 0), val = hit ? idx.v : u_zero();
            ctx.assign_region_smart({Constant(0), Witness(ind_val, OP_IND, R(2), 0, 0, (uint32_t)i), idx, Witness(val, OP_IND_VAL, R(2), 0, 0, (uint32_t)i),
                                     Constant(f_neg(u_from(i))), Witness(ind_val, OP_IND, R(2), 0, 0, (uint32_t)i), Constant(0)},
                                    {0, 3}, {{1, 5}});
            if (i == 0) idx = Existing(ctx.get(-5));
            const Assigned cell = ctx.get(-2);
            assert_bit(ctx, cell);
            ind.push_back(cell);
        }
        return ind;
    }
    // | 0 | a0 | ind0 | s0 | a1 | ind1 | s1 | ...  with s the running selection
    Assigned select_by_indicator(Context &ctx, const std::vector<QCell> &a, const std::vector<Assigned> &ind) const {
        if (a.size() != ind.size()) throw std::runtime_error("select_by_indicator: length mismatch");
        std::vector<QCell> cells;
        std::vector<int> gates;
        cells.reserve(1 + 3 * a.size());
        cells.push_back(Constant(0));
        U256 s = u_zero();
        for (size_t i = 0; i < a.size(); ++i) {
            if (!u_is_zero(ind[i].v)) s = a[i].v;
            gates.push_back((int)(3 * i));
            cells.push_back(a[i]);
            cells.push_back(Existing(ind[i]));
            cells.push_back(Witness(s, OP_SELECT_IND, R((int)(3 * i + 1)), R((int)(3 * i + 2)), R((int)(3 * i))));
        }
        ctx.assign_region(cells, gates);
        return ctx.last();
    }
    Assigned select_from_idx(Context &ctx, const std::vector<QCell> &cells, const QCell &idx) const {
        const std::vector<Assigned> ind = idx_to_indicator(ctx, idx, cells.size());
        return select_by_indicator(ctx, cells, ind);
    }
};

// ------------------------------------------------------------------------------------------- RangeChip
// halo2-base gates/range.rs `RangeInstructions for RangeChip` (RangeStrategy::Vertical) [UPSTREAM, recalled]
struct RangeChip {
    GateChip gate;
    unsigned lookup_bits;
    std::vector<U256> limb_bases;      // 2^(lookup_bits i)
    explicit RangeChip(unsigned lb) : lookup_bits(lb) {
        if (lb == 0 || lb > 28) throw std::runtime_error("lookup_bits out of range");
        for (unsigned i = 0; i * lb < 254; ++i) limb_bases.push_back(f_from_u(u_pow2(i * lb)));
    }
    void range_check(Context &ctx, const Assigned &a, unsigned range_bits) const {
        const unsigned k = (range_bits + lookup_bits - 1) / lookup_bits, rem_bits = range_bits % lookup_bits;
        if (k > limb_bases.size()) throw std::runtime_error("range_check: too many limbs");
        if (k == 1) {
            ctx.cells_to_lookup.push_back(a.off);
        } else {
            std::vector<QCell> limbs, bases;
            for (unsigned i = 0; i < k; ++i) {      // decompose_fe_to_u64_limbs
                limbs.push_back(Witness(u_low_bits(u_shr(a.v, i * lookup_bits), lookup_bits), OP_BITS, a.off, 0, 0, i * lookup_bits | lookup_bits << 8));
                bases.push_back(Constant(limb_bases[i]));
            }
            const int64_t row = (int64_t)ctx.advice.size();
            const Assigned acc = gate.inner_product(ctx, limbs, bases);
            ctx.constrain_equal(a, acc);
            ctx.cells_to_lookup.push_back(row);
            for (unsigned i = 0; i + 1 < k; ++i) ctx.cells_to_lookup.push_back(row + 1 + 3 * (int64_t)i);
        }
        if (rem_bits == 1) {
            gate.assert_bit(ctx, ctx.get(ctx.cells_to_lookup.back()));
        } else if (rem_bits > 1) {
            const Assigned check = gate.mul(ctx, Existing(ctx.get(ctx.cells_to_lookup.back())), Constant(gate.pow_of_two[lookup_bits - rem_bits]));
            ctx.cells_to_lookup.push_back(check.off);
        }
    }
    // | a + 2^bits - b | b | 1 | a + 2^bits | -2^bits | 1 | a |, then the first cell is range-checked
    void check_less_than(Context &ctx, const QCell &a, const QCell &b, unsigned num_bits) const {
        const U256 pow = gate.pow_of_two[num_bits], shift_a = f_add(pow, a.v);
        ctx.assign_region({Witness(f_sub(shift_a, b.v), OP_SUB, R(3), R(1)), b, Constant(1), Witness(shift_a, OP_SUB, R(6), R(4)), Constant(f_neg(pow)),
                           Constant(1), a},
                          {0, 3});
        range_check(ctx, ctx.get(-7), num_bits);
    }
    void check_big_less_than_safe(Context &ctx, const Assigned &a, const U256 &b) const {
        const unsigned range_bits = ((unsigned)u_bits(b) + lookup_bits - 1) / lookup_bits * lookup_bits;
        range_check(ctx, a, range_bits);
        check_less_than(ctx, Existing(a), Constant(f_from_u(b)), range_bits);
    }
    Assigned is_less_than(Context &ctx, const QCell &a, const QCell &b, unsigned num_bits) const {
        const unsigned k = (num_bits + lookup_bits - 1) / lookup_bits, padded_bits = k * lookup_bits;
        const U256 pow = gate.pow_of_two[padded_bits], shift_a = f_add(pow, a.v);
        ctx.assign_region({Witness(f_sub(shift_a, b.v), OP_SUB, R(3), R(1)), b, Constant(1), Witness(shift_a, OP_SUB, R(6), R(4)), Constant(f_neg(pow)),
                           Constant(1), a},
                          {0, 3});
        range_check(ctx, ctx.get(-7), padded_bits + lookup_bits);
        return gate.is_zero(ctx, ctx.get(ctx.cells_to_lookup.back()));      // the top limb is zero iff a < b
    }
    // a = b q + r with a constant divisor: | r | b | q | a |
    std::pair<Assigned, Assigned> div_mod(Context &ctx, const QCell &a, const U256 &b, unsigned a_num_bits) const {
        U256 q, r;
        u_divmod(a.v, b, q, r);
        unsigned e = 0;      // the recorder replays division by a power of two only (the only divisors these chips use)
        if (ctx.recording) {
            e = (unsigned)u_bits(b) - 1;
            if (u_is_zero(b) || u_pow2(e) != b) throw std::runtime_error("recording: div_mod by a constant that is not a power of two");
        }
        ctx.assign_region({Witness(r, OP_BITS, R(3), 0, 0, e << 8), Constant(f_from_u(b)), Witness(q, OP_BITS, R(3), 0, 0, e | 256u << 8), a}, {0});
        const Assigned rem = ctx.get(-4), div = ctx.get(-2);
        U256 bound, unused;
        u_divmod(u_pow2(a_num_bits), b, bound, unused);
        bound = u_add(bound, u_from(1));
        check_big_less_than_safe(ctx, div, bound);
        check_big_less_than_safe(ctx, rem, b);
        return {div, rem};
    }
    // a = b q + r with a witness divisor
    std::pair<Assigned, Assigned> div_mod_var(Context &ctx, const QCell &a, const QCell &b, unsigned a_num_bits, unsigned b_num_bits) const {
        U256 q, r;
        u_divmod(a.v, b.v, q, r);
        ctx.assign_region({Witness(r, OP_DIV_R, R(3), R(1)), b, Witness(q, OP_DIV_Q, R(3), R(1)), a}, {0});
        const Assigned rem = ctx.get(-4), div = ctx.get(-2);
        range_check(ctx, div, a_num_bits);
        range_check(ctx, rem, b_num_bits);
        check_less_than(ctx, Existing(rem), b, b_num_bits);
        return {div, rem};
    }
};

}  // namespace zk
}  // namespace h2v
