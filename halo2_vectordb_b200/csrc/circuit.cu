// circuit.cu -- C ABI of the circuit builder (SURVEY.md 8(f) row 4): the reference's chips run on the host, their
// execution trace is laid out into the columns that h2v_pk_load / h2v_create_proof consume.  No device code here.
//
// Restates [UPSTREAM halo2-base v0.3.0 gates/builder.rs, recalled] as reached from /root/reference/src/scaffold/mod.rs:
//   * `GateThreadBuilder::config(k, minimum_rows)` (mod.rs:388): columns = ceil(cells / (2^k - minimum_rows));
//   * `assign_all` (mod.rs:391-399 RangeCircuitBuilder::{mock, keygen, prover}): cells go down one advice column after the
//     other, a column is left when a gate would cross `max_rows` (the cell is repeated on row 0 of the next column and
//     tied by a copy constraint -- these rows are the pinned `break_points`), lookup cells are copied into the
//     lookup-advice columns, every distinct constant gets one fixed cell;
//   * halo2 `permutation::keygen::Assembly::copy` for the cycles behind the sigma polynomials;
//   * `RangeWithInstanceCircuitBuilder`: one instance column tied to the `make_public` cells (mod.rs:400, 427-433).
#include <algorithm>
#include <memory>
#include <chrono>
#include <thread>

#include "internal.hpp"
#include "zk_chips.hpp"

using namespace h2v;
using namespace h2v::zk;

struct h2v_builder {
    Context ctx;
    FixedPointChip fp;
    DistanceChip dist;
    VectorDBChip vdb;
    std::unique_ptr<PoseidonChip3> poseidon;
    std::vector<int64_t> instances;      // `make_public`
    uint32_t n_inputs = 0;               // values passed to h2v_builder_assign_witnesses
    h2v_builder(unsigned p, unsigned lb) : fp(p, lb), dist(fp), vdb(fp) {
        // the trace of a real circuit has 10^7 - 10^8 cells: reserve address space once (untouched pages cost nothing) instead
        // of re-copying gigabytes at every doubling of the vectors; H2V_TRACE_RESERVE = cells (0 = let them grow)
        const char *e = getenv("H2V_TRACE_RESERVE");
        const size_t cells = e ? (size_t)atoll(e) : ((size_t)1 << 26);
        if (cells) {
            try {
                ctx.advice.reserve(cells);
                ctx.selector.reserve(cells);
                ctx.advice_eq.reserve(cells / 3);
                ctx.constant_eq.reserve(cells / 3);
                ctx.cells_to_lookup.reserve(cells / 6);
            } catch (const std::bad_alloc &) {      // no address space to spare: grow on demand
            }
        }
    }
};

struct h2v_layout {
    uint32_t k, minimum_rows, lookup_bits;
    uint32_t n_gate_advice, n_lookup_advice, n_const_fixed, n_instances;
    std::vector<uint32_t> break_points;
    // columns, Montgomery form, 2^k x 4 limbs each
    std::vector<std::vector<uint64_t>> advice;      // gate columns, then lookup-advice columns
    std::vector<std::vector<uint64_t>> fixed;       // [0] lookup table, [1 ..] constants, then one selector per gate column
    std::vector<std::vector<uint64_t>> sigma;       // permutation columns: constants, advice (gate, lookup), instance
    std::vector<uint64_t> instance;                 // n_instances x 4
    std::vector<const uint64_t *> ptrs[3];
};

namespace {

template <class F> int guarded(F &&f) {
    try {
        return f();
    } catch (const std::exception &e) {      // upstream panics
        return failf(H2V_EINVAL, "%s", e.what());
    }
}
inline U256 from_abi(const uint64_t *p) { return as_u(frh::from_mont(frh::load(p))); }
inline void to_abi(uint64_t *p, const U256 &v) { frh::store(p, frh::to_mont(as_fr(v))); }
Assigned cell(const h2v_builder *b, int64_t off) {
    if (off < 0 || off >= (int64_t)b->ctx.advice.size()) throw std::runtime_error("cell index out of range");
    return Assigned{b->ctx.advice[(size_t)off], off};
}
std::vector<Assigned> cells(const h2v_builder *b, const int64_t *p, size_t n) {
    std::vector<Assigned> out;
    out.reserve(n);
    for (size_t i = 0; i < n; ++i) out.push_back(cell(b, p[i]));
    return out;
}
DistanceFn distance_fn(const h2v_builder *b, int kind) {
    const DistanceChip *d = &b->dist;
    switch (kind) {
        case H2V_DISTANCE_EUCLIDEAN: return [d](Context &c, const std::vector<Assigned> &x, const std::vector<Assigned> &y) { return d->euclidean_distance(c, x, y); };
        case H2V_DISTANCE_COSINE: return [d](Context &c, const std::vector<Assigned> &x, const std::vector<Assigned> &y) { return d->cosine_distance(c, x, y); };
        case H2V_DISTANCE_HAMMING: return [d](Context &c, const std::vector<Assigned> &x, const std::vector<Assigned> &y) { return d->hamming_distance(c, x, y); };
        case H2V_DISTANCE_MANHATTAN: return [d](Context &c, const std::vector<Assigned> &x, const std::vector<Assigned> &y) { return d->manhattan_distance(c, x, y); };
    }
    throw std::runtime_error("unknown distance");
}
U256 f_pow(const U256 &base, const U256 &e) {
    Fr64 acc = frh::ONE, b = frh::to_mont(as_fr(base));
    for (int i = u_bits(e) - 1; i >= 0; --i) {
        acc = frh::sqr(acc);
        if (u_bit(e, (unsigned)i)) acc = frh::mul(acc, b);
    }
    return as_u(frh::from_mont(acc));
}
template <class F> void parallel_for(size_t n, F &&f) {
    const unsigned hw = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
    const size_t nt = std::min<size_t>(hw, n ? n : 1);
    std::vector<std::thread> th;
    for (size_t t = 0; t < nt; ++t)
        th.emplace_back([&, t]() {
            for (size_t i = t; i < n; i += nt) f(i);
        });
    for (auto &x : th) x.join();
}

// halo2 permutation keygen `Assembly`: union of cycles, smaller merged into larger, in the order of the copy() calls
struct Cycles {
    size_t rows;
    // flattened (column * rows + row); 40 M entries each for the kmeans circuit: allocated raw and initialised by all cores
    // (first-touch page faults are most of the cost of a serial fill)
    std::unique_ptr<uint32_t[]> mapping, aux, sizes;
    Cycles(size_t cols, size_t rows_) : rows(rows_), mapping(new uint32_t[cols * rows_]), aux(new uint32_t[cols * rows_]), sizes(new uint32_t[cols * rows_]) {
        uint32_t *m = mapping.get(), *a = aux.get(), *z = sizes.get();
        parallel_for(cols, [&](size_t c) {
            for (size_t i = c * rows_; i < (c + 1) * rows_; ++i) {
                m[i] = a[i] = (uint32_t)i;
                z[i] = 1;
            }
        });
    }
    void copy(size_t lc, size_t lr, size_t rc, size_t rr) {
        uint32_t left = (uint32_t)(lc * rows + lr), right = (uint32_t)(rc * rows + rr);
        uint32_t left_cycle = aux[left], right_cycle = aux[right];
        if (left_cycle == right_cycle) return;
        if (sizes[left_cycle] < sizes[right_cycle]) {
            std::swap(left_cycle, right_cycle);
            std::swap(left, right);
        }
        sizes[left_cycle] += sizes[right_cycle];
        uint32_t i = right_cycle;
        do {
            aux[i] = left_cycle;
            i = mapping[i];
        } while (i != right_cycle);
        std::swap(mapping[left], mapping[right]);
    }
};

// Where assign_all puts each trace cell: the gate columns with their break points, and the lookup-advice columns
struct Placement {
    size_t n, max_rows, num_advice, num_lookup;
    std::vector<uint32_t> pos_col, pos_row;
    struct Break {
        size_t cell;
        uint32_t col, row;
    };
    std::vector<Break> breaks;      // the cell closing column col at row `row` is repeated on row 0 of column col + 1
    std::vector<uint32_t> break_points;
    // the j-th lookup cell: (advice column, row)
    std::pair<size_t, size_t> lookup_pos(size_t j) const { return {num_advice + j / max_rows, j % max_rows}; }
};
void place(const h2v_builder *b, uint32_t k, uint32_t minimum_rows, Placement &P) {
    const Context &ctx = b->ctx;
    if (k < 3 || k > 26) throw std::runtime_error("k out of range");
    const size_t n = (size_t)1 << k;
    if (minimum_rows >= n) throw std::runtime_error("minimum_rows >= 2^k");
    if (b->fp.lookup_bits >= k) throw std::runtime_error("LOOKUP_BITS needs to be less than DEGREE");      // mod.rs:367
    const size_t max_rows = n - minimum_rows;
    // ---- config(): column counts
    const size_t total_advice = ctx.advice.size(), total_lookup = ctx.cells_to_lookup.size();
    const size_t num_advice = (total_advice + max_rows - 1) / max_rows;
    P.n = n;
    P.max_rows = max_rows;
    P.num_advice = num_advice;
    P.num_lookup = (total_lookup + max_rows - 1) / max_rows;
    // ---- assign_all, first loop: positions and break points of the trace down the gate columns
    P.pos_col.resize(total_advice);
    P.pos_row.resize(total_advice);
    size_t gate_index = 0, row = 0;
    for (size_t i = 0; i < total_advice; ++i) {
        if (gate_index >= num_advice) throw std::runtime_error("NOT ENOUGH ADVICE COLUMNS IN PHASE 0. Perhaps blinding factors were not taken into account.");
        P.pos_col[i] = (uint32_t)gate_index;
        P.pos_row[i] = (uint32_t)row;
        const bool q = ctx.selector[i] != 0;
        if ((q && row + 4 > max_rows) || row >= max_rows - 1) {
            // the cell closes this column; it is repeated on row 0 of the next one (where its gate, if any, lives)
            // and tied to the original, which stays the cell's position for the equality constraints
            P.break_points.push_back((uint32_t)row);
            P.breaks.push_back(Placement::Break{i, (uint32_t)gate_index, (uint32_t)row});
            row = 0;
            ++gate_index;
            if (gate_index >= num_advice) throw std::runtime_error("NOT ENOUGH ADVICE COLUMNS IN PHASE 0. Perhaps blinding factors were not taken into account.");
        }
        ++row;
    }
}

int do_layout(const h2v_builder *b, uint32_t k, uint32_t minimum_rows, h2v_layout *L) {
    const Context &ctx = b->ctx;
    const bool timing = getenv("H2V_LAYOUT_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto tick = [&](const char *what) {
        if (!timing) return;
        auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "layout: %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(t - t_last).count());
        t_last = t;
    };
    Placement pl;
    place(b, k, minimum_rows, pl);
    const size_t n = pl.n, max_rows = pl.max_rows, total_advice = ctx.advice.size();
    const size_t num_advice = pl.num_advice, num_lookup = pl.num_lookup;
    L->k = k;
    L->minimum_rows = minimum_rows;
    L->lookup_bits = b->fp.lookup_bits;
    std::unordered_map<U256, std::pair<uint32_t, uint32_t>, U256Hash> assigned_constants;
    std::vector<U256> const_order;
    for (const auto &ce : ctx.constant_eq)
        if (assigned_constants.emplace(ce.first, std::make_pair(0u, 0u)).second) const_order.push_back(ce.first);
    const size_t num_fixed = (const_order.size() + n - 1) >> k;
    L->n_gate_advice = (uint32_t)num_advice;
    L->n_lookup_advice = (uint32_t)num_lookup;
    L->n_const_fixed = (uint32_t)num_fixed;
    L->n_instances = (uint32_t)b->instances.size();
    if (L->n_instances > max_rows) throw std::runtime_error("too many public inputs");
    const size_t A = num_advice + num_lookup, F = 1 + num_fixed + num_advice;
    // permutation columns: constants, gate advice, lookup advice, instance
    const size_t P = num_fixed + A + 1;
    const size_t pc_const = 0, pc_adv = num_fixed, pc_inst = num_fixed + A;
    // columns are written as canonical limbs first and converted to Montgomery form in place at the end
    L->advice.assign(A, std::vector<uint64_t>());
    L->fixed.assign(F, std::vector<uint64_t>());
    parallel_for(A + F, [&](size_t j) { (j < A ? L->advice[j] : L->fixed[j - A]).assign(n * 4, 0); });      // 2.3 GB at kmeans size: first touch by all cores
    auto put = [](std::vector<uint64_t> &col, size_t row, const U256 &v) { memcpy(&col[4 * row], v.l, 32); };
    std::vector<std::vector<uint64_t>> &adv = L->advice, &fix = L->fixed;
    tick("allocate columns");
    Cycles cyc(P, n);
    tick("cycles init");
    // ---- assign_all, first loop: the trace down the gate columns
    const std::vector<uint32_t> &pos_col = pl.pos_col, &pos_row = pl.pos_row;
    L->break_points = pl.break_points;
    {
        // the values and selector cells by all cores
        const size_t parts = 64;
        parallel_for(parts, [&](size_t part) {
            const size_t i0 = total_advice * part / parts, i1 = total_advice * (part + 1) / parts;
            for (size_t i = i0; i < i1; ++i) {
                put(adv[pos_col[i]], pos_row[i], ctx.advice[i]);
                if (ctx.selector[i]) put(fix[1 + num_fixed + pos_col[i]], pos_row[i], u_from(1));
            }
        });
        for (const Placement::Break &bk : pl.breaks) {
            put(adv[bk.col + 1], 0, ctx.advice[bk.cell]);
            if (ctx.selector[bk.cell]) {        // the gate starts on the repeated cell, not on the closing one
                put(fix[1 + num_fixed + bk.col], bk.row, u_from(0));
                put(fix[1 + num_fixed + bk.col + 1], 0, u_from(1));
            }
            cyc.copy(pc_adv + bk.col + 1, 0, pc_adv + bk.col, bk.row);
        }
    }
    tick("trace -> gate columns");
    // constants: one fixed cell per distinct value, column-cyclic
    if (!const_order.empty() && num_fixed == 0) throw std::runtime_error("no fixed column for constants");
    {
        size_t fixed_col = 0, fixed_off = 0;
        for (const U256 &c : const_order) {
            put(fix[1 + fixed_col], fixed_off, c);
            assigned_constants[c] = std::make_pair((uint32_t)fixed_col, (uint32_t)fixed_off);
            if (++fixed_col >= num_fixed) {
                fixed_col = 0;
                ++fixed_off;
            }
        }
    }
    // ---- second loop: equality constraints, then the lookup copies
    for (const auto &e : ctx.advice_eq)
        cyc.copy(pc_adv + pos_col[(size_t)e.first], pos_row[(size_t)e.first], pc_adv + pos_col[(size_t)e.second], pos_row[(size_t)e.second]);
    tick("advice equalities");
    if (timing) fprintf(stderr, "layout: %zu advice equalities, %zu constant equalities, %zu lookup cells\n", ctx.advice_eq.size(), ctx.constant_eq.size(), ctx.cells_to_lookup.size());
    for (const auto &e : ctx.constant_eq) {
        const auto fc = assigned_constants[e.first];
        cyc.copy(pc_const + fc.first, fc.second, pc_adv + pos_col[(size_t)e.second], pos_row[(size_t)e.second]);
    }
    for (size_t j = 0; j < ctx.cells_to_lookup.size(); ++j) {
        const size_t off = (size_t)ctx.cells_to_lookup[j];
        const auto lp = pl.lookup_pos(j);
        put(adv[lp.first], lp.second, ctx.advice[off]);
        cyc.copy(pc_adv + pos_col[off], pos_row[off], pc_adv + lp.first, lp.second);
    }
    tick("constant + lookup copies");
    // lookup table 0 .. 2^lookup_bits - 1 (the remaining rows hold the default 0)
    for (size_t i = 0; i < ((size_t)1 << b->fp.lookup_bits); ++i) put(fix[0], i, u_from(i));
    // instance column
    L->instance.assign((size_t)L->n_instances * 4, 0);
    for (size_t i = 0; i < b->instances.size(); ++i) {
        const size_t off = (size_t)b->instances[i];
        to_abi(&L->instance[4 * i], ctx.advice[off]);
        cyc.copy(pc_adv + pos_col[off], pos_row[off], pc_inst, i);
    }
    // ---- Montgomery columns, sigma = delta^column * omega^row of the image
    U256 t_exp, rem_;
    u_divmod(u_sub(f_modulus(), u_from(1)), u_pow2(28), t_exp, rem_);
    const U256 root = f_pow(u_from(7), t_exp);                       // Fr::ROOT_OF_UNITY
    const U256 omega = f_pow(root, u_pow2(28 - k));
    const Fr64 delta = frh::to_mont(as_fr(f_pow(u_from(7), u_pow2(28))));      // Fr::DELTA
    std::vector<Fr64> wp(n), dp(P);
    wp[0] = frh::ONE;
    const Fr64 om = frh::to_mont(as_fr(omega));
    for (size_t i = 1; i < n; ++i) wp[i] = frh::mul(wp[i - 1], om);
    dp[0] = frh::ONE;
    for (size_t c = 1; c < P; ++c) dp[c] = frh::mul(dp[c - 1], delta);
    L->sigma.assign(P, std::vector<uint64_t>());
    tick("tables, powers");
    parallel_for(A + F + P, [&](size_t j) {
        if (j < A + F) {
            std::vector<uint64_t> &col = j < A ? L->advice[j] : L->fixed[j - A];
            for (size_t i = 0; i < n; ++i) {
                uint64_t *p = &col[4 * i];
                if (p[0] | p[1] | p[2] | p[3]) frh::store(p, frh::to_mont(frh::load(p)));
            }
        } else {
            const size_t c = j - A - F;
            std::vector<uint64_t> &dst = L->sigma[c];
            dst.resize(n * 4);
            for (size_t i = 0; i < n; ++i) {
                const uint32_t m = cyc.mapping[c * n + i];
                frh::store(&dst[4 * i], frh::mul(dp[m / n], wp[m % n]));
            }
        }
    });
    tick("montgomery + sigma");
    for (int kind = 0; kind < 3; ++kind) {
        auto &cols = kind == 0 ? L->advice : kind == 1 ? L->fixed : L->sigma;
        L->ptrs[kind].clear();
        for (auto &c : cols) L->ptrs[kind].push_back(c.data());
    }
    return H2V_OK;
}

// The witness program of a recording: copies resolved to their roots, the cells no input reaches folded to their recorded
// values, the others sorted by level; the gather map from the layout's advice positions and instances to them.
void make_plan(const h2v_builder *b, uint32_t k, uint32_t minimum_rows, WitnessPlan &W) {
    const Context &ctx = b->ctx;
    if (!ctx.recording) throw std::runtime_error("witness_program: the builder is not a recording builder (h2v_builder_new_recording)");
    Placement pl;
    place(b, k, minimum_rows, pl);
    if (b->instances.size() > pl.max_rows) throw std::runtime_error("too many public inputs");
    const size_t N = ctx.advice.size();
    if (N >= WREF_POOL) throw std::runtime_error("witness_program: too many cells");
    const std::vector<Rule> &rules = ctx.rules;
    auto nargs = [](uint8_t kind) {
        switch (kind) {
            case OP_ADD: case OP_SUB: case OP_MUL: case OP_OR: case OP_DIV_Q: case OP_DIV_R: return 2;
            case OP_MUL_ADD: case OP_SELECT_IND: return 3;
            default: return 1;
        }
    };
    std::vector<uint32_t> root(N);
    for (size_t i = 0; i < N; ++i) {
        const Rule &r = rules[i];
        if (r.kind == RULE_NONE || r.kind >= RULE_KINDS) throw std::runtime_error("witness_program: cell " + std::to_string(i) + " has no rule");
        if (r.kind == RULE_COPY) {
            if (r.a < 0 || (size_t)r.a >= i) throw std::runtime_error("witness_program: cell " + std::to_string(i) + " copies a later cell");
            root[i] = root[(size_t)r.a];
        } else {
            root[i] = (uint32_t)i;
        }
        const int64_t ops[3] = {r.a, r.b, r.c};
        if (r.kind >= OP_ADD)
            for (int j = 0; j < nargs(r.kind); ++j)
                if (ops[j] < 0 || (size_t)ops[j] >= N || (size_t)ops[j] == i) throw std::runtime_error("witness_program: cell " + std::to_string(i) + " has a bad operand");
    }
    // level of each root: -1 folded (no input reaches it), 0 input, else 1 + the deepest computed operand
    const int32_t UNSEEN = -2, VISITING = -3;
    std::vector<int32_t> level(N, UNSEEN);
    auto operands = [&](size_t i, uint32_t *o) {      // the operands' roots (unused operands are cell 0, never read)
        const int na = nargs(rules[i].kind);
        o[0] = root[(size_t)rules[i].a];
        o[1] = na > 1 ? root[(size_t)rules[i].b] : 0;
        o[2] = na > 2 ? root[(size_t)rules[i].c] : 0;
    };
    std::vector<uint32_t> stack;
    uint32_t n_levels = 0;
    for (size_t i0 = 0; i0 < N; ++i0) {
        if (root[i0] != i0 || level[i0] != UNSEEN) continue;
        stack.push_back((uint32_t)i0);
        while (!stack.empty()) {
            const uint32_t i = stack.back();
            const Rule &r = rules[i];
            if (level[i] >= -1) {      // pushed twice
                stack.pop_back();
                continue;
            }
            if (r.kind == RULE_INPUT || r.kind == RULE_CONST) {
                level[i] = r.kind == RULE_INPUT ? 0 : -1;
                stack.pop_back();
                continue;
            }
            uint32_t o[3];
            operands(i, o);
            const int na = nargs(r.kind);
            bool ready = true;
            for (int j = 0; j < na; ++j)
                if (level[o[j]] == UNSEEN) {
                    if (ready) level[i] = VISITING;
                    ready = false;
                    stack.push_back(o[j]);
                } else if (level[o[j]] == VISITING) {
                    throw std::runtime_error("witness_program: cell " + std::to_string(i) + " depends on itself");
                }
            if (!ready) continue;
            int32_t lv = -1;
            for (int j = 0; j < na; ++j) lv = std::max(lv, level[o[j]]);
            level[i] = lv < 0 ? -1 : lv + 1;
            n_levels = std::max(n_levels, (uint32_t)std::max(level[i], 0));
            stack.pop_back();
        }
    }
    // slots: inputs by their index, then the computed cells level by level (trace order within a level)
    W.k = k;
    W.n_cells = N;
    W.n_inputs = b->n_inputs;
    W.n_levels = n_levels;
    W.level_start.assign((size_t)n_levels + 2, 0);
    for (size_t i = 0; i < N; ++i)
        if (root[i] == i && level[i] > 0) ++W.level_start[(size_t)level[i] + 1];
    for (size_t l = 1; l < W.level_start.size(); ++l) W.level_start[l] += W.level_start[l - 1];
    W.level_start.erase(W.level_start.begin());      // level l (1-based) occupies [level_start[l - 1], level_start[l])
    const size_t n_computed = W.level_start.back();
    std::vector<uint32_t> slot(N, WREF_ZERO), fill(W.level_start.begin(), W.level_start.end() - 1);
    W.inputs.assign(W.n_inputs * 4, 0);
    for (size_t i = 0; i < N; ++i) {
        if (root[i] != i) continue;
        if (level[i] == 0) {
            slot[i] = rules[i].imm;
            to_abi(&W.inputs[4 * (size_t)rules[i].imm], ctx.advice[i]);
        } else if (level[i] > 0) {
            slot[i] = (uint32_t)(W.n_inputs + fill[(size_t)level[i] - 1]++);
        }
    }
    if (W.n_inputs + n_computed >= WREF_POOL) throw std::runtime_error("witness_program: too many cells");
    std::unordered_map<uint32_t, uint32_t> pool_of;
    auto ref = [&](uint32_t c) -> uint32_t {      // c: a root cell
        if (slot[c] != WREF_ZERO) return slot[c];
        if (u_is_zero(ctx.advice[c])) return WREF_ZERO;
        auto it = pool_of.emplace(c, (uint32_t)(W.pool.size() / 4));
        if (it.second) W.pool.insert(W.pool.end(), ctx.advice[c].l, ctx.advice[c].l + 4);
        return WREF_POOL | it.first->second;
    };
    W.kind_counts.assign(RULE_KINDS, 0);
    W.rules.resize(n_computed);
    W.cell_of.resize(n_computed);
    for (size_t i = 0; i < N; ++i) {
        if (root[i] != i || level[i] <= 0) continue;
        const Rule &r = rules[i];
        if (r.imm >= (1u << 24)) throw std::runtime_error("witness_program: immediate out of range");
        uint32_t o[3], rr[3] = {WREF_ZERO, WREF_ZERO, WREF_ZERO};
        operands(i, o);
        for (int j = 0; j < nargs(r.kind); ++j) rr[j] = ref(o[j]);
        const size_t s_ = slot[i] - W.n_inputs;
        W.rules[s_] = WitnessRule{rr[0], rr[1], rr[2], (uint32_t)r.kind | r.imm << 8};
        W.cell_of[s_] = i;
        ++W.kind_counts[r.kind];
    }
    // gather map: the layout's advice columns (gate columns with the break repeats, lookup columns), then the instances
    const size_t n = pl.n, A = pl.num_advice + pl.num_lookup;
    W.n_adv_cols = A;
    W.n_instances = b->instances.size();
    W.map.assign(A * n + W.n_instances, WREF_ZERO);
    for (size_t i = 0; i < N; ++i) W.map[(size_t)pl.pos_col[i] * n + pl.pos_row[i]] = ref(root[i]);
    for (const Placement::Break &bk : pl.breaks) W.map[(size_t)(bk.col + 1) * n] = ref(root[bk.cell]);
    for (size_t j = 0; j < ctx.cells_to_lookup.size(); ++j) {
        const auto lp = pl.lookup_pos(j);
        W.map[lp.first * n + lp.second] = ref(root[(size_t)ctx.cells_to_lookup[j]]);
    }
    for (size_t i = 0; i < W.n_instances; ++i) W.map[A * n + i] = ref(root[(size_t)b->instances[i]]);
}

}  // namespace

extern "C" {

int h2v_builder_new_recording(uint32_t precision_bits, uint32_t lookup_bits, h2v_builder_t *out) {
    H2V_TRY(h2v_builder_new(precision_bits, lookup_bits, out));
    (*out)->ctx.recording = true;
    return H2V_OK;
}
int h2v_witness_program_new(h2v_builder_t b, uint32_t k, uint32_t minimum_rows, h2v_witness_program_t *out) {
    if (!b || !out) return failf(H2V_EINVAL, "witness_program_new: NULL argument");
    WitnessPlan plan;
    H2V_TRY(guarded([&]() {
        make_plan(b, k, minimum_rows, plan);
        return (int)H2V_OK;
    }));
    return witness_program_make(std::move(plan), out);
}

int h2v_builder_new(uint32_t precision_bits, uint32_t lookup_bits, h2v_builder_t *out) {
    if (!out) return failf(H2V_EINVAL, "builder_new: out is NULL");
    return guarded([&]() {
        *out = new h2v_builder(precision_bits, lookup_bits);
        return (int)H2V_OK;
    });
}
void h2v_builder_free(h2v_builder_t b) { delete b; }

int h2v_builder_quantize(h2v_builder_t b, const double *x, size_t n, uint64_t *out) {
    if (!b || (n && (!x || !out))) return failf(H2V_EINVAL, "quantize: NULL argument");
    for (size_t i = 0; i < n; ++i) to_abi(out + 4 * i, b->fp.quantization(x[i]));
    return H2V_OK;
}
int h2v_builder_dequantize(h2v_builder_t b, const uint64_t *x, size_t n, double *out) {
    if (!b || (n && (!x || !out))) return failf(H2V_EINVAL, "dequantize: NULL argument");
    for (size_t i = 0; i < n; ++i) out[i] = b->fp.dequantization(from_abi(x + 4 * i));
    return H2V_OK;
}
int h2v_builder_assign_witnesses(h2v_builder_t b, const uint64_t *values, size_t n, int64_t *cells_out) {
    if (!b || (n && (!values || !cells_out))) return failf(H2V_EINVAL, "assign_witnesses: NULL argument");
    for (size_t i = 0; i < n; ++i) cells_out[i] = b->ctx.load_witness(Witness(from_abi(values + 4 * i), RULE_INPUT, 0, 0, 0, b->n_inputs++)).off;
    return H2V_OK;
}
int h2v_builder_load_constant(h2v_builder_t b, const uint64_t value[4], int64_t *cell_out) {
    if (!b || !value || !cell_out) return failf(H2V_EINVAL, "load_constant: NULL argument");
    *cell_out = b->ctx.load_constant(from_abi(value)).off;
    return H2V_OK;
}
int h2v_builder_cell_values(h2v_builder_t b, const int64_t *cells_, size_t n, uint64_t *out) {
    if (!b || (n && (!cells_ || !out))) return failf(H2V_EINVAL, "cell_values: NULL argument");
    return guarded([&]() {
        for (size_t i = 0; i < n; ++i) to_abi(out + 4 * i, cell(b, cells_[i]).v);
        return (int)H2V_OK;
    });
}
int h2v_builder_make_public(h2v_builder_t b, const int64_t *cells_, size_t n) {
    if (!b || (n && !cells_)) return failf(H2V_EINVAL, "make_public: NULL argument");
    return guarded([&]() {
        for (size_t i = 0; i < n; ++i) b->instances.push_back(cell(b, cells_[i]).off);
        return (int)H2V_OK;
    });
}

int h2v_builder_call(h2v_builder_t b, int op, const int64_t *in, size_t n_in, int64_t *out) {
    if (!b || !out || (n_in && !in)) return failf(H2V_EINVAL, "builder_call: NULL argument");
    return guarded([&]() {
        Context &c = b->ctx;
        const FixedPointChip &fp = b->fp;
        auto need = [&](size_t k_) {
            if (n_in != k_) throw std::runtime_error("builder_call: wrong number of cells for this operation");
        };
        auto q = [&](size_t i) { return Existing(cell(b, in[i])); };
        Assigned r{};
        switch (op) {
            case H2V_FP_QADD: need(2); r = fp.qadd(c, q(0), q(1)); break;
            case H2V_FP_QSUB: need(2); r = fp.qsub(c, q(0), q(1)); break;
            case H2V_FP_QMUL: need(2); r = fp.qmul(c, q(0), q(1)); break;
            case H2V_FP_QDIV: need(2); r = fp.qdiv(c, q(0), q(1)); break;
            case H2V_FP_QMOD: need(2); r = fp.qmod(c, q(0), q(1)); break;
            case H2V_FP_QPOW: need(2); r = fp.qpow(c, q(0), q(1)); break;
            case H2V_FP_QMAX: need(2); r = fp.qmax(c, q(0), q(1)); break;
            case H2V_FP_QMIN: need(2); r = fp.qmin(c, q(0), q(1)); break;
            case H2V_FP_BIT_XOR: need(2); r = fp.bit_xor(c, q(0), q(1)); break;
            case H2V_FP_COND_NEG: need(2); r = fp.cond_neg(c, q(0), cell(b, in[1])); break;
            case H2V_FP_NEG: need(1); r = fp.neg(c, q(0)); break;
            case H2V_FP_QABS: need(1); r = fp.qabs(c, q(0)); break;
            case H2V_FP_IS_NEG: need(1); r = fp.is_neg(c, q(0)); break;
            case H2V_FP_SIGN: need(1); r = fp.sign(c, q(0)); break;
            case H2V_FP_CLIP: need(1); r = fp.clip(c, q(0)); break;
            case H2V_FP_QEXP2: need(1); r = fp.qexp2(c, q(0)); break;
            case H2V_FP_QLOG2: need(1); r = fp.qlog2(c, q(0)); break;
            case H2V_FP_QEXP: need(1); r = fp.qexp(c, q(0)); break;
            case H2V_FP_QLOG: need(1); r = fp.qlog(c, q(0)); break;
            case H2V_FP_QSQRT: need(1); r = fp.qsqrt(c, q(0)); break;
            case H2V_FP_QSIN: need(1); r = fp.qsin(c, q(0)); break;
            case H2V_FP_QCOS: need(1); r = fp.qcos(c, q(0)); break;
            case H2V_FP_QTAN: need(1); r = fp.qtan(c, q(0)); break;
            case H2V_FP_QSINH: need(1); r = fp.qsinh(c, q(0)); break;
            case H2V_FP_QCOSH: need(1); r = fp.qcosh(c, q(0)); break;
            case H2V_FP_QTANH: need(1); r = fp.qtanh(c, q(0)); break;
            case H2V_FP_QSUM: r = fp.qsum(c, existing(cells(b, in, n_in))); break;
            case H2V_FP_INNER_PRODUCT: {
                if (n_in % 2) throw std::runtime_error("assertion failed: a.len() == b.len()");
                r = fp.inner_product(c, existing(cells(b, in, n_in / 2)), existing(cells(b, in + n_in / 2, n_in / 2)));
                break;
            }
            case H2V_FP_POLYNOMIAL: {      // in[0] = x, in[1..] = coefficients, highest degree first
                if (n_in < 2) throw std::runtime_error("polynomial: no coefficients");
                r = fp.polynomial(c, q(0), existing(cells(b, in + 1, n_in - 1)));
                break;
            }
            case H2V_DISTANCE_EUCLIDEAN:
            case H2V_DISTANCE_COSINE:
            case H2V_DISTANCE_HAMMING:
            case H2V_DISTANCE_MANHATTAN: {
                if (n_in % 2) throw std::runtime_error("assertion failed: a.len() == b.len()");
                r = distance_fn(b, op)(c, cells(b, in, n_in / 2), cells(b, in + n_in / 2, n_in / 2));
                break;
            }
            default: throw std::runtime_error("builder_call: unknown operation");
        }
        *out = r.off;
        return (int)H2V_OK;
    });
}

int h2v_builder_nearest_vector(h2v_builder_t b, int distance, const int64_t *query, const int64_t *vectors, size_t n_vec, size_t dim,
                               int64_t *indicator_out, int64_t *result_out) {
    if (!b || !query || !vectors || !indicator_out || !result_out) return failf(H2V_EINVAL, "nearest_vector: NULL argument");
    return guarded([&]() {
        std::vector<std::vector<Assigned>> vs;
        for (size_t v = 0; v < n_vec; ++v) vs.push_back(cells(b, vectors + v * dim, dim));
        const auto res = b->vdb.nearest_vector(b->ctx, cells(b, query, dim), vs, distance_fn(b, distance));
        for (size_t i = 0; i < n_vec; ++i) indicator_out[i] = res.first[i].off;
        for (size_t i = 0; i < dim; ++i) result_out[i] = res.second[i].off;
        return (int)H2V_OK;
    });
}
int h2v_builder_poseidon_new(h2v_builder_t b, uint32_t t, uint32_t rate, uint32_t r_f, uint32_t r_p) {
    if (!b) return failf(H2V_EINVAL, "poseidon_new: NULL builder");
    if (t != 3 || rate != 2) return failf(H2V_EINVAL, "poseidon_new: only T = 3, RATE = 2 (examples/query.rs:27-28) is built");
    if (r_f < 2 || r_f % 2 || r_p < 1) return failf(H2V_EINVAL, "poseidon_new: bad round numbers");
    return guarded([&]() {
        b->poseidon.reset(new PoseidonChip3(b->ctx, (int)r_f, (int)r_p));
        return (int)H2V_OK;
    });
}
int h2v_builder_poseidon_hash(h2v_builder_t b, const int64_t *in, size_t n, int64_t *out) {
    if (!b || !out || (n && !in)) return failf(H2V_EINVAL, "poseidon_hash: NULL argument");
    if (!b->poseidon) return failf(H2V_EINVAL, "poseidon_hash: call h2v_builder_poseidon_new first");
    return guarded([&]() {
        b->poseidon->clear();
        b->poseidon->update(cells(b, in, n));
        *out = b->poseidon->squeeze(b->ctx, b->fp.gate()).off;
        return (int)H2V_OK;
    });
}
int h2v_builder_merkle_commitment(h2v_builder_t b, const int64_t *vectors, size_t n_vec, size_t dim, int64_t *root_out) {
    if (!b || !vectors || !root_out) return failf(H2V_EINVAL, "merkle_commitment: NULL argument");
    if (!b->poseidon) return failf(H2V_EINVAL, "merkle_commitment: call h2v_builder_poseidon_new first");
    return guarded([&]() {
        std::vector<std::vector<Assigned>> vs;
        for (size_t v = 0; v < n_vec; ++v) vs.push_back(cells(b, vectors + v * dim, dim));
        *root_out = b->vdb.merkle_commitment(b->ctx, *b->poseidon, vs).off;
        return (int)H2V_OK;
    });
}
int h2v_builder_kmeans(h2v_builder_t b, int distance, const int64_t *vectors, size_t n_vec, size_t dim, uint32_t K, uint32_t I,
                       int64_t *centroids_out, int64_t *indicators_out) {
    if (!b || !vectors || !centroids_out || !indicators_out) return failf(H2V_EINVAL, "kmeans: NULL argument");
    return guarded([&]() {
        std::vector<std::vector<Assigned>> vs;
        for (size_t v = 0; v < n_vec; ++v) vs.push_back(cells(b, vectors + v * dim, dim));
        const auto res = b->vdb.kmeans(b->ctx, vs, K, I, distance_fn(b, distance));
        for (size_t c = 0; c < K; ++c)
            for (size_t d = 0; d < dim; ++d) centroids_out[c * dim + d] = res.first[c][d].off;
        for (size_t v = 0; v < res.second.size(); ++v)
            for (size_t c = 0; c < K; ++c) indicators_out[v * K + c] = res.second[v][c].off;
        return (int)H2V_OK;
    });
}

int h2v_builder_stats(h2v_builder_t b, uint64_t out[4]) {
    if (!b || !out) return failf(H2V_EINVAL, "builder_stats: NULL argument");
    std::unordered_map<U256, int, U256Hash> distinct;
    for (const auto &ce : b->ctx.constant_eq) distinct.emplace(ce.first, 0);
    out[0] = b->ctx.advice.size();
    out[1] = b->ctx.cells_to_lookup.size();
    out[2] = distinct.size();
    out[3] = b->instances.size();
    return H2V_OK;
}
int h2v_builder_config(h2v_builder_t b, uint32_t k, uint32_t minimum_rows, uint32_t out[3]) {
    if (!b || !out) return failf(H2V_EINVAL, "builder_config: NULL argument");
    if (k < 1 || k > 30 || minimum_rows >= (1ull << k)) return failf(H2V_EINVAL, "builder_config: bad k / minimum_rows");
    uint64_t st[4];
    h2v_builder_stats(b, st);
    const uint64_t max_rows = (1ull << k) - minimum_rows;
    out[0] = (uint32_t)((st[0] + max_rows - 1) / max_rows);
    out[1] = (uint32_t)((st[1] + max_rows - 1) / max_rows);
    out[2] = (uint32_t)((st[2] + (1ull << k) - 1) >> k);
    return H2V_OK;
}
int h2v_builder_trace(h2v_builder_t b, uint64_t *advice_out, uint8_t *selector_out, int64_t *lookup_out) {
    if (!b) return failf(H2V_EINVAL, "builder_trace: NULL builder");
    const Context &c = b->ctx;
    if (advice_out)
        for (size_t i = 0; i < c.advice.size(); ++i) memcpy(advice_out + 4 * i, c.advice[i].l, 32);      // canonical
    if (selector_out) memcpy(selector_out, c.selector.data(), c.selector.size());
    if (lookup_out) memcpy(lookup_out, c.cells_to_lookup.data(), c.cells_to_lookup.size() * sizeof(int64_t));
    return H2V_OK;
}

int h2v_builder_layout(h2v_builder_t b, uint32_t k, uint32_t minimum_rows, h2v_layout_t *out) {
    if (!b || !out) return failf(H2V_EINVAL, "builder_layout: NULL argument");
    std::unique_ptr<h2v_layout> L(new h2v_layout());
    const int rc = guarded([&]() { return do_layout(b, k, minimum_rows, L.get()); });
    if (rc) return rc;
    *out = L.release();
    return H2V_OK;
}
void h2v_layout_free(h2v_layout_t l) { delete l; }
int h2v_layout_info(h2v_layout_t l, uint32_t out[8]) {
    if (!l || !out) return failf(H2V_EINVAL, "layout_info: NULL argument");
    out[0] = l->k;
    out[1] = l->n_gate_advice;
    out[2] = l->n_lookup_advice;
    out[3] = l->n_const_fixed;
    out[4] = l->n_instances;
    out[5] = (uint32_t)l->break_points.size();
    out[6] = l->lookup_bits;
    out[7] = l->minimum_rows;
    return H2V_OK;
}
int h2v_layout_columns(h2v_layout_t l, int kind, const uint64_t *const **cols_out, size_t *n_cols) {
    if (!l || !cols_out || !n_cols) return failf(H2V_EINVAL, "layout_columns: NULL argument");
    if (kind < 0 || kind > 2) return failf(H2V_EINVAL, "layout_columns: kind must be 0 (advice), 1 (fixed) or 2 (sigma)");
    *cols_out = l->ptrs[kind].data();
    *n_cols = l->ptrs[kind].size();
    return H2V_OK;
}
int h2v_layout_instance(h2v_layout_t l, const uint64_t **out, size_t *n) {
    if (!l || !out || !n) return failf(H2V_EINVAL, "layout_instance: NULL argument");
    *out = l->instance.data();
    *n = l->n_instances;
    return H2V_OK;
}
int h2v_layout_break_points(h2v_layout_t l, uint32_t *out, size_t cap, size_t *n) {
    if (!l || !n) return failf(H2V_EINVAL, "layout_break_points: NULL argument");
    *n = l->break_points.size();
    if (out) {
        if (cap < l->break_points.size()) return failf(H2V_EINVAL, "layout_break_points: buffer too small");
        memcpy(out, l->break_points.data(), l->break_points.size() * sizeof(uint32_t));
    }
    return H2V_OK;
}

}  // extern "C"
