// mock.cu -- h2v_mock_prover: halo2's MockProver checks (every gate, lookup and copy constraint of a laid-out circuit) on
// the device, for the constraint-system shape the prover takes (include/h2v.h, "mock prover").
//
// Every check is data-parallel over (column, row), so each one is a kernel that sets a flag bit; the bits are laid out in
// the order the failures are reported (gates, lookups, permutation; column; row; the four permutation checks of a cell),
// and an ordered compaction (popcount per group of 1024 bits, exclusive scan, emit) writes the first `cap` of them.
//   gates        one thread per (gate, row), straight from the selector and advice columns in Lagrange form
//   lookups      each distinct table column's usable rows are sorted once (sort_canonical_dev, the lookup argument's
//                bitonic sort), then one binary search per input cell
//   permutation  sigma = delta^c2 w^r2 is decoded per cell: v^n (k squarings) is looked up among the n_perm values
//                delta^(c n) (distinct: delta's order is the odd part of r - 1), then v delta^-c2 in a hash table of the 2^k
//                values w^r.  "Image already hit by an earlier cell" is one atomicMin of the visiting cell's linear index per
//                image, and a second pass flags every visitor that is not the minimum, so the output does not depend on
//                the order threads run in.
// Device memory: the columns, 4 bytes per permutation cell (the atomicMin array), the flag bits and 1/32 of them for the
// compaction, w^r with its hash table (40 bytes per row) and the sorted tables (32 bytes per row and table).
#include <cuda_runtime.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <vector>

#include "h2v.h"
#include "internal.hpp"
#include "ff.cuh"

using namespace h2v;

namespace {

typedef FrP Fr;
constexpr uint32_t EMPTY = 0xffffffffu;
constexpr uint32_t GROUP_WORDS = 32;      // flag words per compaction group (1024 flags)

__device__ __forceinline__ fe ld(const fe *p) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    uint4 a = q[0], b = q[1];
    fe r;
    r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
    r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
    return r;
}
// x mod r for any 256-bit x (x < 2^256 < 6r): subtract 4r, 2r, r where possible.  Montgomery limbs reduced this way compare
// equal exactly when the field elements are equal.
__device__ __forceinline__ fe canon(fe v) {
#pragma unroll
    for (int sh = 2; sh >= 0; --sh) {
        uint32_t m[8], d[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = (uint32_t)(((uint64_t)Fr::m(i) << sh) | (i ? ((uint64_t)Fr::m(i - 1) >> (32 - sh)) : 0));
        const uint32_t bw = raw_sub(d, v.v, m);
#pragma unroll
        for (int i = 0; i < 8; ++i) v.v[i] = bw ? v.v[i] : d[i];
    }
    return v;
}
__device__ __forceinline__ fe ldc(const fe *p) { return canon(ld(p)); }
__device__ __forceinline__ void set_flag(uint32_t *bits, uint64_t b) { atomicOr(bits + (b >> 5), 1u << (b & 31)); }

// open-addressing hash tables of field elements (canonical Montgomery limbs): slot -> index into a value array
H2V_HD uint32_t slot_of(const fe &x, uint32_t mask) { return ((x.v[0] * 0x9e3779b1u) ^ x.v[7]) & mask; }
__device__ __forceinline__ uint32_t hash_find(const uint32_t *tab, uint32_t mask, const fe *vals, const fe &x) {
    for (uint32_t s = slot_of(x, mask);; s = (s + 1) & mask) {
        const uint32_t e = tab[s];
        if (e == EMPTY || fe_eq(ld(vals + e), x)) return e;
    }
}

// ------------------------------------------------------------------ gates
// gate j (grid.y), row i: q = sel[j][i] != 0  ->  flag j * n + i when i + 3 >= u or a + a(w) a(w^2) - a(w^3) != 0
__global__ void __launch_bounds__(256) mock_gate_kernel(const fe *const *sel, const fe *const *adv, uint32_t n, uint32_t u, uint32_t *bits) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y;
    if (i >= n || fe_is_zero(ldc(sel[j] + i))) return;
    bool bad = i + 3 >= u;
    if (!bad) {
        const fe *a = adv[j] + i;
        bad = !fe_is_zero(fe_sub<Fr>(fe_add<Fr>(ldc(a), fe_mul<Fr>(ldc(a + 1), ldc(a + 2))), ldc(a + 3)));
    }
    if (bad) set_flag(bits, (uint64_t)j * n + i);
}

// ------------------------------------------------------------------ lookups
// lookup l (grid.y), usable row i: the canonical input value must occur in its table's sorted keys[tmap[l]][0 .. u)
__global__ void __launch_bounds__(256) mock_lookup_kernel(const fe *const *inputs, const fe *keys, const uint32_t *tmap, uint32_t u,
                                                          uint32_t n_pad, uint32_t n, uint64_t base, uint32_t *bits) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y;
    if (i >= u) return;
    const fe v = fe_from_mont<Fr>(ld(inputs[l] + i));
    const fe *T = keys + (size_t)tmap[l] * n_pad;
    uint32_t lo = 0, hi = u;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (key_less(ld(T + mid), v)) lo = mid + 1;
        else hi = mid;
    }
    if (lo == u || !key_eq(ld(T + lo), v)) set_flag(bits, base + (uint64_t)l * n + i);
}

// ------------------------------------------------------------------ permutation
struct PermArgs {
    const fe *const *sigma;      // n_perm sigma columns
    const fe *const *vals;       // the n_perm permuted columns (advice / fixed / instance padded with zeros)
    const fe *col_vals;          // delta^(c n), c < n_perm
    const fe *dinv;              // delta^-c
    const uint32_t *col_tab;     // hash table over col_vals
    const fe *omega_pows;        // w^r, r < n
    const uint32_t *row_tab;     // hash table over omega_pows
    uint32_t col_mask, row_mask, k, n, u;
    uint32_t *first;             // per image (c2 n + r2): the least linear index c n + r of a cell mapped onto it
    uint32_t *bits;
    uint64_t base;               // flag of check s (0..3) of cell (c, r): base + 4 (c n + r) + s
};
__device__ __forceinline__ bool decode(const PermArgs &a, const fe &v, uint32_t &c2, uint32_t &r2) {
    fe y = v;
    for (uint32_t t = 0; t < a.k; ++t) y = fe_sqr<Fr>(y);
    c2 = hash_find(a.col_tab, a.col_mask, a.col_vals, y);
    if (c2 == EMPTY) return false;
    r2 = hash_find(a.row_tab, a.row_mask, a.omega_pows, fe_mul<Fr>(v, ld(a.dinv + c2)));
    return r2 != EMPTY;
}
// w^r for every row and its hash table (the table has 2n slots, so probing ends)
__global__ void __launch_bounds__(256) mock_omega_table_kernel(fe omega, uint32_t n, fe *omega_pows, uint32_t *tab, uint32_t mask) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const fe w = fe_pow_small<Fr>(omega, r);
    uint4 *q = reinterpret_cast<uint4 *>(omega_pows + r);
    q[0] = make_uint4(w.v[0], w.v[1], w.v[2], w.v[3]);
    q[1] = make_uint4(w.v[4], w.v[5], w.v[6], w.v[7]);
    for (uint32_t s = slot_of(w, mask);; s = (s + 1) & mask)
        if (atomicCAS(tab + s, EMPTY, r) == EMPTY) break;
}
// pass 1, column c (grid.y), row i: flag a sigma value that does not decode, else offer the cell's index to its image
__global__ void __launch_bounds__(256) mock_perm_first_kernel(PermArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (i >= a.n) return;
    const uint32_t lin = c * a.n + i;
    uint32_t c2, r2;
    if (!decode(a, ldc(a.sigma[c] + i), c2, r2)) set_flag(a.bits, a.base + 4ull * lin);
    else atomicMin(a.first + c2 * a.n + r2, lin);
}
// pass 2: the image was hit by an earlier cell; a copy into an unusable row; a copy between different values
__global__ void __launch_bounds__(256) mock_perm_check_kernel(PermArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (i >= a.n) return;
    const uint32_t lin = c * a.n + i;
    uint32_t c2, r2;
    if (!decode(a, ldc(a.sigma[c] + i), c2, r2)) return;
    const uint32_t img = c2 * a.n + r2;
    const uint64_t f = a.base + 4ull * lin;
    if (a.first[img] != lin) set_flag(a.bits, f + 1);
    if (img == lin) return;
    if (i >= a.u || r2 >= a.u) set_flag(a.bits, f + 2);
    if (!fe_eq(ldc(a.vals[c] + i), ldc(a.vals[c2] + r2))) set_flag(a.bits, f + 3);
}

// ------------------------------------------------------------------ ordered compaction
__global__ void __launch_bounds__(256) mock_count_kernel(const uint32_t *bits, uint64_t n_words, uint32_t n_groups, uint32_t *counts) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const uint64_t w0 = (uint64_t)g * GROUP_WORDS, w1 = min(w0 + GROUP_WORDS, n_words);
    uint32_t s = 0;
    for (uint64_t w = w0; w < w1; ++w) s += __popc(bits[w]);
    counts[g] = s;
}
struct Sections {
    uint32_t n, u;
    uint64_t lookup_base, perm_base;         // first flag of the lookup / permutation section
    const uint32_t *gate_adv, *lookup_in;    // the advice column of each gate / lookup
};
// group g writes its flags, in order, to out[offs[g] ...] as long as the index is below cap
__global__ void __launch_bounds__(256) mock_emit_kernel(const uint32_t *bits, uint64_t n_words, uint32_t n_groups, const uint32_t *offs,
                                                        uint32_t cap, Sections s, PermArgs a, h2v_mock_failure_t *out) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    uint32_t idx = offs[g];
    const uint64_t w0 = (uint64_t)g * GROUP_WORDS, w1 = min(w0 + GROUP_WORDS, n_words);
    for (uint64_t w = w0; w < w1 && idx < cap; ++w) {
        for (uint32_t m = bits[w]; m && idx < cap; m &= m - 1, ++idx) {
            const uint64_t b = w * 32 + (__ffs(m) - 1);
            h2v_mock_failure_t f;
            if (b < s.lookup_base) {
                f.column = (uint32_t)(b / s.n);
                f.row = (uint32_t)(b % s.n);
                f.kind = f.row + 3 >= s.u ? H2V_MOCK_GATE_UNUSABLE : H2V_MOCK_GATE;
                f.other_column = s.gate_adv[f.column];
                f.other_row = f.row;
            } else if (b < s.perm_base) {
                f.column = (uint32_t)((b - s.lookup_base) / s.n);
                f.row = (uint32_t)((b - s.lookup_base) % s.n);
                f.kind = H2V_MOCK_LOOKUP;
                f.other_column = s.lookup_in[f.column];
                f.other_row = f.row;
            } else {
                const uint64_t p = b - s.perm_base;
                const uint32_t check = (uint32_t)(p & 3), lin = (uint32_t)(p >> 2);
                f.column = lin / s.n;
                f.row = lin % s.n;
                f.kind = H2V_MOCK_SIGMA_NOT_DELTA_OMEGA + check;
                f.other_column = f.other_row = EMPTY;
                if (check) decode(a, ldc(a.sigma[f.column] + f.row), f.other_column, f.other_row);
            }
            out[idx] = f;
        }
    }
}

// ------------------------------------------------------------------ host side
thread_local double t_last_ms[2] = {0, 0};

double now_ms() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
fe host_fe(uint64_t x) {
    fe c = fe_zero();
    c.v[0] = (uint32_t)x;
    c.v[1] = (uint32_t)(x >> 32);
    return fe_to_mont<Fr>(c);
}
uint32_t pow2_at_least(uint64_t x) {
    uint32_t p = 1;
    while (p < x) p <<= 1;
    return p;
}

// the device buffers and stream of one call, freed on every return path
struct MockCall {
    DevBuf cols, tabs, keys, first, rows, bits, scan, out;
    cudaStream_t st = nullptr;
    ~MockCall() {
        for (DevBuf *b : {&cols, &tabs, &keys, &first, &rows, &bits, &scan, &out}) b->release();
        if (st) cudaStreamDestroy(st);
    }
};

int mock_run(const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma, const uint64_t *const *advice,
             const uint64_t *const *instances, const uint32_t *instance_len, h2v_mock_failure_t *failures_out, size_t cap,
             uint64_t *n_failures) {
    const uint32_t k = cs->k, n = 1u << k, u = n - (cs->blinding_factors + 1);
    const uint32_t G = cs->n_gates, L = cs->n_lookups, P = cs->n_perm, A = cs->n_advice, F = cs->n_fixed, I = cs->n_instance;
    const uint64_t lookup_base = (uint64_t)G * n, perm_base = lookup_base + (uint64_t)L * n, n_flags = perm_base + 4ull * P * n;
    MockCall m;
    H2V_CU(cudaStreamCreateWithFlags(&m.st, cudaStreamNonBlocking));
    cudaStream_t st = m.st;

    // columns: advice, fixed, sigma, instance (zero-padded to n rows)
    const double t0 = now_ms();
    const size_t n_cols = (size_t)A + F + P + I;
    H2V_TRY(m.cols.ensure(std::max<size_t>(n_cols, 1) * n * sizeof(fe)));
    fe *adv_d = m.cols.as<fe>(), *fix_d = adv_d + (size_t)A * n, *sig_d = fix_d + (size_t)F * n, *inst_d = sig_d + (size_t)P * n;
    for (uint32_t c = 0; c < A; ++c) H2V_CU(cudaMemcpyAsync(adv_d + (size_t)c * n, advice[c], n * sizeof(fe), cudaMemcpyHostToDevice, st));
    for (uint32_t c = 0; c < F; ++c) H2V_CU(cudaMemcpyAsync(fix_d + (size_t)c * n, fixed[c], n * sizeof(fe), cudaMemcpyHostToDevice, st));
    for (uint32_t c = 0; c < P; ++c) H2V_CU(cudaMemcpyAsync(sig_d + (size_t)c * n, sigma[c], n * sizeof(fe), cudaMemcpyHostToDevice, st));
    if (I) H2V_CU(cudaMemsetAsync(inst_d, 0, (size_t)I * n * sizeof(fe), st));
    for (uint32_t c = 0; c < I; ++c)
        if (instance_len[c]) H2V_CU(cudaMemcpyAsync(inst_d + (size_t)c * n, instances[c], instance_len[c] * sizeof(fe), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaStreamSynchronize(st));
    const double t1 = now_ms();

    // small tables: column pointers, the column index of each gate / lookup, the distinct lookup tables, the permutation's
    // delta^(c n), delta^-c and their hash table
    std::vector<const fe *> ptrs;
    for (uint32_t j = 0; j < G; ++j) ptrs.push_back(fix_d + (size_t)cs->gate_selector[j] * n);
    for (uint32_t j = 0; j < G; ++j) ptrs.push_back(adv_d + (size_t)cs->gate_advice[j] * n);
    for (uint32_t l = 0; l < L; ++l) ptrs.push_back(adv_d + (size_t)cs->lookup_input[l] * n);
    std::vector<uint32_t> tmap(L), tcols;
    for (uint32_t l = 0; l < L; ++l) {
        auto it = std::find(tcols.begin(), tcols.end(), cs->lookup_table[l]);
        tmap[l] = (uint32_t)(it - tcols.begin());
        if (it == tcols.end()) tcols.push_back(cs->lookup_table[l]);
    }
    for (uint32_t t : tcols) ptrs.push_back(fix_d + (size_t)t * n);
    for (uint32_t c = 0; c < P; ++c) ptrs.push_back(sig_d + (size_t)c * n);
    for (uint32_t c = 0; c < P; ++c) {
        const uint32_t idx = cs->perm_index[c];
        ptrs.push_back(cs->perm_kind[c] == 0 ? adv_d + (size_t)idx * n : cs->perm_kind[c] == 1 ? fix_d + (size_t)idx * n : inst_d + (size_t)idx * n);
    }
    const uint32_t col_slots = pow2_at_least(2ull * std::max(P, 1u));
    std::vector<fe> pvals(2 * (size_t)P);          // delta^(c n), then delta^-c
    std::vector<uint32_t> col_tab(col_slots, EMPTY);
    {
        const fe delta = fe_pow_u64<Fr>(host_fe(7), 1ull << 28);     // Fr::DELTA = GENERATOR^(2^S)
        const fe dn = fe_pow_u64<Fr>(delta, n), dinv = fe_inv<Fr>(delta);
        fe a = fe_one<Fr>(), b = fe_one<Fr>();
        for (uint32_t c = 0; c < P; ++c) {
            pvals[c] = a;
            pvals[P + c] = b;
            for (uint32_t s = slot_of(a, col_slots - 1);; s = (s + 1) & (col_slots - 1))
                if (col_tab[s] == EMPTY) {
                    col_tab[s] = c;
                    break;
                }
            a = fe_mul<Fr>(a, dn);
            b = fe_mul<Fr>(b, dinv);
        }
    }
    std::vector<uint32_t> idx32(cs->gate_advice, cs->gate_advice + G);
    idx32.insert(idx32.end(), cs->lookup_input, cs->lookup_input + L);
    idx32.insert(idx32.end(), tmap.begin(), tmap.end());
    idx32.insert(idx32.end(), col_tab.begin(), col_tab.end());
    const size_t ptr_bytes = (ptrs.size() * sizeof(void *) + 15) & ~(size_t)15, fe_bytes = pvals.size() * sizeof(fe);   // fe: 16-byte aligned
    H2V_TRY(m.tabs.ensure(ptr_bytes + fe_bytes + idx32.size() * sizeof(uint32_t) + 64));
    char *tb = m.tabs.as<char>();
    H2V_CU(cudaMemcpyAsync(tb, ptrs.data(), ptrs.size() * sizeof(void *), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(tb + ptr_bytes, pvals.data(), fe_bytes, cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(tb + ptr_bytes + fe_bytes, idx32.data(), idx32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    const fe *const *d_ptrs = reinterpret_cast<const fe *const *>(tb);
    const fe *const *d_sel = d_ptrs, *const *d_gadv = d_ptrs + G, *const *d_lin = d_gadv + G, *const *d_tabs = d_lin + L;
    const fe *const *d_sigma = d_tabs + tcols.size(), *const *d_vals = d_sigma + P;
    const fe *d_pvals = reinterpret_cast<const fe *>(tb + ptr_bytes);
    const uint32_t *d_gate_adv = reinterpret_cast<const uint32_t *>(tb + ptr_bytes + fe_bytes), *d_lookup_in = d_gate_adv + G;
    const uint32_t *d_tmap = d_lookup_in + L, *d_col_tab = d_tmap + L;

    // flags (one bit each, zeroed) and the compaction's counts
    const uint64_t n_words = (n_flags + 31) / 32;
    const uint32_t n_groups = (uint32_t)((n_words + GROUP_WORDS - 1) / GROUP_WORDS);
    const uint32_t n_tiles = (n_groups + 2047) / 2048;
    H2V_TRY(m.bits.ensure(std::max<uint64_t>(n_words, 1) * sizeof(uint32_t)));
    H2V_TRY(m.scan.ensure(((size_t)3 * n_groups + n_tiles + 1) * sizeof(uint32_t)));
    uint32_t *bits = m.bits.as<uint32_t>(), *counts = m.scan.as<uint32_t>(), *offs = counts + n_groups, *scratch = offs + n_groups;
    uint32_t *tiles = scratch + n_groups, *total = tiles + n_tiles;
    H2V_CU(cudaMemsetAsync(bits, 0, n_words * sizeof(uint32_t), st));

    if (G) {
        mock_gate_kernel<<<dim3((n + 255) / 256, G), 256, 0, st>>>(d_sel, d_gadv, n, u, bits);
        H2V_LAUNCHED();
    }
    if (L) {
        const uint32_t n_pad = pow2_at_least(u);
        H2V_TRY(m.keys.ensure(tcols.size() * n_pad * sizeof(fe)));
        H2V_TRY(sort_canonical_dev(st, d_tabs, (uint32_t)tcols.size(), u, n_pad, m.keys.as<fe>()));
        mock_lookup_kernel<<<dim3((u + 255) / 256, L), 256, 0, st>>>(d_lin, m.keys.as<fe>(), d_tmap, u, n_pad, n, lookup_base, bits);
        H2V_LAUNCHED();
    }
    PermArgs pa{};
    pa.sigma = d_sigma;
    pa.vals = d_vals;
    pa.col_vals = d_pvals;
    pa.dinv = d_pvals + P;
    pa.col_tab = d_col_tab;
    pa.col_mask = col_slots - 1;
    pa.k = k;
    pa.n = n;
    pa.u = u;
    pa.bits = bits;
    pa.base = perm_base;
    if (P) {
        H2V_TRY(m.first.ensure((size_t)P * n * sizeof(uint32_t)));
        H2V_TRY(m.rows.ensure((size_t)n * sizeof(fe) + 2 * (size_t)n * sizeof(uint32_t)));
        fe *omega_pows = m.rows.as<fe>();
        uint32_t *row_tab = reinterpret_cast<uint32_t *>(omega_pows + n);
        H2V_CU(cudaMemsetAsync(m.first.p, 0xff, (size_t)P * n * sizeof(uint32_t), st));
        H2V_CU(cudaMemsetAsync(row_tab, 0xff, 2 * (size_t)n * sizeof(uint32_t), st));
        // w = GENERATOR^((r - 1) / 2^k), the 2^k-th root of unity EvaluationDomain::new(_, k) uses
        uint32_t e[8];
        for (int i = 0; i < 8; ++i) e[i] = Fr::m(i);
        e[0] -= 1;
        for (int i = 0; i < 8; ++i) e[i] = (e[i] >> k) | (i < 7 ? e[i + 1] << (32 - k) : 0);
        const fe omega = fe_pow<Fr>(host_fe(7), e);
        mock_omega_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(omega, n, omega_pows, row_tab, 2 * n - 1);
        H2V_LAUNCHED();
        pa.omega_pows = omega_pows;
        pa.row_tab = row_tab;
        pa.row_mask = 2 * n - 1;
        pa.first = m.first.as<uint32_t>();
        mock_perm_first_kernel<<<dim3((n + 255) / 256, P), 256, 0, st>>>(pa);
        H2V_LAUNCHED();
        mock_perm_check_kernel<<<dim3((n + 255) / 256, P), 256, 0, st>>>(pa);
        H2V_LAUNCHED();
    }

    uint32_t tot = 0;
    if (n_groups) {
        mock_count_kernel<<<(n_groups + 255) / 256, 256, 0, st>>>(bits, n_words, n_groups, counts);
        H2V_LAUNCHED();
        H2V_TRY(scan_u32_dev(st, counts, n_groups, offs, tiles, scratch, total));
        H2V_CU(cudaMemcpyAsync(&tot, total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        H2V_CU(cudaStreamSynchronize(st));
    }
    const uint32_t n_out = (uint32_t)std::min<uint64_t>(cap, tot);
    if (n_out) {
        H2V_TRY(m.out.ensure((size_t)n_out * sizeof(h2v_mock_failure_t)));
        const Sections s{n, u, lookup_base, perm_base, d_gate_adv, d_lookup_in};
        mock_emit_kernel<<<(n_groups + 255) / 256, 256, 0, st>>>(bits, n_words, n_groups, offs, n_out, s, pa, m.out.as<h2v_mock_failure_t>());
        H2V_LAUNCHED();
        H2V_CU(cudaMemcpyAsync(failures_out, m.out.p, (size_t)n_out * sizeof(h2v_mock_failure_t), cudaMemcpyDeviceToHost, st));
    }
    H2V_CU(cudaStreamSynchronize(st));
    *n_failures = tot;
    t_last_ms[0] = t1 - t0;
    t_last_ms[1] = now_ms() - t1;
    return H2V_OK;
}

}  // namespace

extern "C" {

int h2v_mock_prover(const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma, const uint64_t *const *advice,
                    const uint64_t *const *instances, const uint32_t *instance_len, h2v_mock_failure_t *failures_out, size_t cap,
                    uint64_t *n_failures) {
    if (!cs || !n_failures || (cap && !failures_out)) return failf(H2V_EINVAL, "mock_prover: NULL argument");
    *n_failures = 0;
    H2V_TRY(check_circuit(cs,
                          !(cs->n_fixed && !fixed) && !(cs->n_perm && !sigma) && !(cs->n_advice && !advice) &&
                              !(cs->n_instance && (!instances || !instance_len)),
                          "mock_prover"));
    const size_t n = (size_t)1 << cs->k;
    for (uint32_t c = 0; c < cs->n_advice; ++c)
        if (!advice[c]) return failf(H2V_EINVAL, "mock_prover: advice column %u is NULL", c);
    for (uint32_t c = 0; c < cs->n_fixed; ++c)
        if (!fixed[c]) return failf(H2V_EINVAL, "mock_prover: fixed column %u is NULL", c);
    for (uint32_t c = 0; c < cs->n_perm; ++c)
        if (!sigma[c]) return failf(H2V_EINVAL, "mock_prover: sigma column %u is NULL", c);
    for (uint32_t c = 0; c < cs->n_instance; ++c) {
        if (instance_len[c] > n) return failf(H2V_EINVAL, "mock_prover: instance column %u has %u values, more than 2^k = %zu", c, instance_len[c], n);
        if (instance_len[c] && !instances[c]) return failf(H2V_EINVAL, "mock_prover: instance column %u is NULL", c);
    }
    if (cs->n_gates > 65535 || cs->n_lookups > 65535 || cs->n_perm > 65535)
        return failf(H2V_EINVAL, "mock_prover: more than 65535 gates, lookups or permutation columns");
    if (((uint64_t)cs->n_gates + cs->n_lookups + 4ull * cs->n_perm) * n >= (1ull << 32))
        return failf(H2V_EINVAL, "mock_prover: (gates + lookups + 4 permutation columns) x 2^k = %llu flags, more than 2^32",
                     (unsigned long long)(((uint64_t)cs->n_gates + cs->n_lookups + 4ull * cs->n_perm) * n));
    if (cudaSetDevice(current_device()) != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ECUDA, "mock_prover: no CUDA device (libh2v has no CPU fallback)");
    }
    return mock_run(cs, fixed, sigma, advice, instances, instance_len, failures_out, cap, n_failures);
}

int h2v_mock_last_ms(double out[2]) {
    if (!out) return failf(H2V_EINVAL, "mock_last_ms: NULL argument");
    out[0] = t_last_ms[0];
    out[1] = t_last_ms[1];
    return H2V_OK;
}

}  // extern "C"
