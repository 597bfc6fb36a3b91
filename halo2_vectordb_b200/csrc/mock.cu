// mock.cu -- h2v_mock_prover and h2v_pk_mock_prover: halo2's MockProver checks (every gate, lookup and copy constraint of a
// laid-out circuit) on the device, for the constraint-system shape the prover takes (include/h2v.h, "mock prover").
//
// Every check is data-parallel over (column, row), so each one is a kernel that sets a flag bit; the bits are laid out in
// the order the failures are reported (gates, lookups, permutation; column; row; the four permutation checks of a cell),
// and an ordered compaction (popcount per group of 1024 bits, exclusive scan, emit) writes the first `cap` of them.
// The checks come in two parts:
//   key tables   (MockKey, built once per key from the fixed and sigma columns)
//                lookups: each distinct table column's usable rows sorted (sort_canonical_dev, the lookup argument's
//                bitonic sort).  permutation: sigma = delta^c2 w^r2 decoded per cell into its image c2 n + r2: v^n (k
//                squarings) is looked up among the n_perm values delta^(c n) (distinct: delta's order is the odd part of
//                r - 1), then v delta^-c2 in a hash table of the 2^k values w^r.  "Image already hit by an earlier cell"
//                is one atomicMin of the visiting cell's linear index per image, and a second pass flags every visitor
//                that is not the minimum, so the output does not depend on the order threads run in.  The permutation's
//                key-only flags (SIGMA_NOT_DELTA_OMEGA, SIGMA_NOT_PERMUTATION, COPY_UNUSABLE) are kept as flag words.
//   witnesses    a batch of B witnesses, witness w on grid.z, each with its own flag section (starting on a compaction
//                group): the key's permutation flag words copied in, then one thread per (gate, row), one binary search
//                per lookup input cell, and one comparison per permutation cell with the value at its image.  One count,
//                one scan and one emit launch serve the batch; emit subtracts the witness's first offset.
// Device memory: the key tables hold 4 bytes and 4 bits per permutation cell and 32 bytes per row of each distinct lookup
// table (building them needs another 4 bytes per permutation cell and 40 bytes per row); a batch needs its witnesses'
// columns, one bit per flag and 1/32 of that for the compaction.
#include <cuda_runtime.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <memory>
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

// The columns of a batch: witness w's advice column c at adv + (w A + c) n, its instance column c (zero-padded to n rows)
// at inst + (w I + c) n; the key's fixed column c at fixed + c n.  Witness w's flags start at bit w * wbits.
struct Batch {
    const fe *adv, *inst, *fixed;
    uint32_t A, I, k, n, u;
    uint64_t wbits;
    uint32_t *bits;
    __device__ const fe *col(uint32_t w, uint32_t kind, uint32_t idx) const {
        return kind == 0 ? adv + ((size_t)w * A + idx) * n : kind == 1 ? fixed + (size_t)idx * n : inst + ((size_t)w * I + idx) * n;
    }
};

// ------------------------------------------------------------------ gates
// gate j (grid.y), row i, witness w (grid.z): q = fixed[sel[j]][i] != 0  ->  flag j * n + i when i + 3 >= u or
// a + a(w) a(w^2) - a(w^3) != 0 with a = advice[gadv[j]]
__global__ void __launch_bounds__(256) mock_gate_kernel(Batch b, const uint32_t *sel, const uint32_t *gadv) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, j = blockIdx.y, w = blockIdx.z;
    if (i >= b.n || fe_is_zero(ldc(b.col(w, 1, sel[j]) + i))) return;
    bool bad = i + 3 >= b.u;
    if (!bad) {
        const fe *a = b.col(w, 0, gadv[j]) + i;
        bad = !fe_is_zero(fe_sub<Fr>(fe_add<Fr>(ldc(a), fe_mul<Fr>(ldc(a + 1), ldc(a + 2))), ldc(a + 3)));
    }
    if (bad) set_flag(b.bits, w * b.wbits + (uint64_t)j * b.n + i);
}

// ------------------------------------------------------------------ lookups
// lookup l (grid.y), usable row i, witness w (grid.z): the canonical value of advice[lin[l]][i] must occur in its table's
// sorted keys[tmap[l]][0 .. u)
__global__ void __launch_bounds__(256) mock_lookup_kernel(Batch b, const uint32_t *lin, const fe *keys, const uint32_t *tmap, uint32_t n_pad,
                                                          uint64_t base) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y, w = blockIdx.z;
    if (i >= b.u) return;
    const fe v = fe_from_mont<Fr>(ld(b.col(w, 0, lin[l]) + i));
    const fe *T = keys + (size_t)tmap[l] * n_pad;
    uint32_t lo = 0, hi = b.u;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (key_less(ld(T + mid), v)) lo = mid + 1;
        else hi = mid;
    }
    if (lo == b.u || !key_eq(ld(T + lo), v)) set_flag(b.bits, w * b.wbits + base + (uint64_t)l * b.n + i);
}

// ------------------------------------------------------------------ permutation
// The key-only part.  Flag s (0..3) of cell (c, r) is bit 4 (c n + r) + s of the permutation section.
struct PermKeyArgs {
    const fe *sigma;             // n_perm sigma columns of n rows
    const fe *col_vals;          // delta^(c n), c < n_perm
    const fe *dinv;              // delta^-c
    const uint32_t *col_tab;     // hash table over col_vals
    const fe *omega_pows;        // w^r, r < n
    const uint32_t *row_tab;     // hash table over omega_pows
    uint32_t col_mask, row_mask, k, n, u;
    uint32_t *img;               // per cell: its image c2 n + r2, or EMPTY
    uint32_t *first;             // per image: the least linear index c n + r of a cell mapped onto it
    uint32_t *bits;              // the permutation section's flags
};
__device__ __forceinline__ bool decode(const PermKeyArgs &a, const fe &v, uint32_t &c2, uint32_t &r2) {
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
// pass 1, column c (grid.y), row i: decode the cell's image; flag a sigma value that does not decode, else offer the
// cell's index to its image
__global__ void __launch_bounds__(256) mock_perm_decode_kernel(PermKeyArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (i >= a.n) return;
    const uint32_t lin = c * a.n + i;
    uint32_t c2, r2;
    if (!decode(a, ldc(a.sigma + (size_t)lin), c2, r2)) {
        a.img[lin] = EMPTY;
        set_flag(a.bits, 4ull * lin);
    } else {
        a.img[lin] = c2 * a.n + r2;
        atomicMin(a.first + c2 * a.n + r2, lin);
    }
}
// pass 2: the image was hit by an earlier cell; a copy into an unusable row
__global__ void __launch_bounds__(256) mock_perm_key_kernel(PermKeyArgs a) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y;
    if (i >= a.n) return;
    const uint32_t lin = c * a.n + i, img = a.img[lin];
    if (img == EMPTY) return;
    if (a.first[img] != lin) set_flag(a.bits, 4ull * lin + 1);
    if (img != lin && (i >= a.u || (img & (a.n - 1)) >= a.u)) set_flag(a.bits, 4ull * lin + 2);
}
// The witness part, column c (grid.y), row i, witness w (grid.z): a copy between different values.  The permutation
// section starts at bit `base` of the witness's flags.
__global__ void __launch_bounds__(256) mock_copy_kernel(Batch b, const uint32_t *img, const uint32_t *pkind, const uint32_t *pidx, uint64_t base) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, c = blockIdx.y, w = blockIdx.z;
    if (i >= b.n) return;
    const uint32_t lin = c * b.n + i, im = img[lin];
    if (im == EMPTY || im == lin) return;
    const uint32_t c2 = im >> b.k, r2 = im & (b.n - 1);
    if (!fe_eq(ldc(b.col(w, pkind[c], pidx[c]) + i), ldc(b.col(w, pkind[c2], pidx[c2]) + r2)))
        set_flag(b.bits, w * b.wbits + base + 4ull * lin + 3);
}

// ------------------------------------------------------------------ ordered compaction
__global__ void __launch_bounds__(256) mock_count_kernel(const uint32_t *bits, uint32_t n_groups, uint32_t *counts) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const uint64_t w0 = (uint64_t)g * GROUP_WORDS;
    uint32_t s = 0;
    for (uint64_t w = w0; w < w0 + GROUP_WORDS; ++w) s += __popc(bits[w]);
    counts[g] = s;
}
struct Sections {
    uint32_t k, n, u, gpw;                   // gpw: compaction groups per witness
    uint64_t lookup_base, perm_base;         // first flag of the lookup / permutation section of a witness
    const uint32_t *gate_adv, *lookup_in;    // the advice column of each gate / lookup
    const uint32_t *img;                     // the image of each permutation cell
};
// group g of witness w = g / gpw writes its flags, in order, to out[w cap + offs[g] - offs[w gpw] ...] while that index is
// below cap
__global__ void __launch_bounds__(256) mock_emit_kernel(const uint32_t *bits, uint32_t n_groups, const uint32_t *offs, uint32_t cap, Sections s,
                                                        h2v_mock_failure_t *out) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const uint32_t wit = g / s.gpw;
    uint32_t idx = offs[g] - offs[(size_t)wit * s.gpw];
    out += (size_t)wit * cap;
    const uint64_t w0 = (uint64_t)g * GROUP_WORDS, wit0 = (uint64_t)wit * s.gpw * GROUP_WORDS;
    for (uint64_t w = w0; w < w0 + GROUP_WORDS && idx < cap; ++w) {
        for (uint32_t m = bits[w]; m && idx < cap; m &= m - 1, ++idx) {
            const uint64_t b = (w - wit0) * 32 + (__ffs(m) - 1);
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
                f.column = lin >> s.k;
                f.row = lin & (s.n - 1);
                f.kind = H2V_MOCK_SIGMA_NOT_DELTA_OMEGA + check;
                f.other_column = f.other_row = EMPTY;
                if (check) {
                    const uint32_t im = s.img[lin];
                    f.other_column = im >> s.k;
                    f.other_row = im & (s.n - 1);
                }
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
uint64_t round_up(uint64_t x, uint64_t m) { return (x + m - 1) / m * m; }

}  // namespace

namespace h2v {

// The key tables.  A witness's flags: gates (G n), lookups (L n), then from the next word on the permutation section
// (4 P n), padded to a whole number of compaction groups.
struct MockKey {
    uint32_t k = 0, n = 0, u = 0, G = 0, L = 0, P = 0, A = 0, I = 0, n_pad = 0;
    uint64_t lookup_base = 0, perm_base = 0, flags = 0, wbits = 0;   // flags: (G + L + 4 P) n, the flags one witness can set
    const fe *fixed = nullptr;                // the key's fixed columns (not owned)
    DevBuf idx;                               // gate_selector, gate_advice (G each), lookup_input, tmap (L each), perm_kind, perm_index (P each)
    DevBuf keys, img, pbits;                  // sorted tables, the image of each permutation cell, the permutation section's key-only flags
    ~MockKey() {
        for (DevBuf *b : {&idx, &keys, &img, &pbits}) b->release();
    }
    const uint32_t *sel() const { return idx.as<uint32_t>(); }
    const uint32_t *gadv() const { return sel() + G; }
    const uint32_t *lin() const { return gadv() + G; }
    const uint32_t *tmap() const { return lin() + L; }
    const uint32_t *pkind() const { return tmap() + L; }
    const uint32_t *pidx() const { return pkind() + P; }
};

void mock_key_free(MockKey *key) { delete key; }

int mock_key_build(cudaStream_t st, const h2v_circuit_t *cs, const fe *fixed, const fe *sigma, MockKey **out) {
    std::unique_ptr<MockKey> key(new MockKey());
    MockKey &K = *key;
    K.k = cs->k;
    K.n = 1u << K.k;
    K.u = K.n - (cs->blinding_factors + 1);
    K.G = cs->n_gates; K.L = cs->n_lookups; K.P = cs->n_perm; K.A = cs->n_advice; K.I = cs->n_instance;
    K.fixed = fixed;
    const uint32_t n = K.n, G = K.G, L = K.L, P = K.P;
    K.lookup_base = (uint64_t)G * n;
    K.perm_base = round_up(K.lookup_base + (uint64_t)L * n, 32);
    K.flags = ((uint64_t)G + L + 4ull * P) * n;
    K.wbits = round_up(K.perm_base + 4ull * P * n, 32 * GROUP_WORDS);

    // index tables, the distinct lookup tables, the permutation's delta^(c n), delta^-c and their hash table
    std::vector<uint32_t> tmap(L), tcols;
    for (uint32_t l = 0; l < L; ++l) {
        auto it = std::find(tcols.begin(), tcols.end(), cs->lookup_table[l]);
        tmap[l] = (uint32_t)(it - tcols.begin());
        if (it == tcols.end()) tcols.push_back(cs->lookup_table[l]);
    }
    std::vector<uint32_t> idx(cs->gate_selector, cs->gate_selector + G);
    idx.insert(idx.end(), cs->gate_advice, cs->gate_advice + G);
    idx.insert(idx.end(), cs->lookup_input, cs->lookup_input + L);
    idx.insert(idx.end(), tmap.begin(), tmap.end());
    idx.insert(idx.end(), cs->perm_kind, cs->perm_kind + P);
    idx.insert(idx.end(), cs->perm_index, cs->perm_index + P);
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
    std::vector<const fe *> tptr;
    for (uint32_t t : tcols) tptr.push_back(fixed + (size_t)t * n);
    H2V_TRY(K.idx.ensure(std::max<size_t>(idx.size(), 1) * sizeof(uint32_t)));
    H2V_CU(cudaMemcpyAsync(K.idx.p, idx.data(), idx.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));

    // what only the build needs: the table pointers, pvals, col_tab, w^r with its hash table and the atomicMin array
    struct Scratch {
        DevBuf small, rows, first;
        ~Scratch() {
            for (DevBuf *b : {&small, &rows, &first}) b->release();
        }
    } tmp;
    const size_t ptr_bytes = (tptr.size() * sizeof(void *) + 15) & ~(size_t)15, fe_bytes = pvals.size() * sizeof(fe);   // fe: 16-byte aligned
    H2V_TRY(tmp.small.ensure(ptr_bytes + fe_bytes + col_tab.size() * sizeof(uint32_t) + 64));
    char *tb = tmp.small.as<char>();
    if (!tptr.empty()) H2V_CU(cudaMemcpyAsync(tb, tptr.data(), tptr.size() * sizeof(void *), cudaMemcpyHostToDevice, st));
    if (fe_bytes) H2V_CU(cudaMemcpyAsync(tb + ptr_bytes, pvals.data(), fe_bytes, cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(tb + ptr_bytes + fe_bytes, col_tab.data(), col_tab.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));

    if (L) {
        K.n_pad = pow2_at_least(K.u);
        H2V_TRY(K.keys.ensure(tcols.size() * K.n_pad * sizeof(fe)));
        H2V_TRY(sort_canonical_dev(st, reinterpret_cast<const fe *const *>(tb), (uint32_t)tcols.size(), K.u, K.n_pad, K.keys.as<fe>()));
    }
    if (P) {
        const size_t cells = (size_t)P * n, pwords = (4 * cells + 31) / 32;
        H2V_TRY(K.img.ensure(cells * sizeof(uint32_t)));
        H2V_TRY(K.pbits.ensure(pwords * sizeof(uint32_t)));
        H2V_TRY(tmp.first.ensure(cells * sizeof(uint32_t)));
        H2V_TRY(tmp.rows.ensure((size_t)n * sizeof(fe) + 2 * (size_t)n * sizeof(uint32_t)));
        fe *omega_pows = tmp.rows.as<fe>();
        uint32_t *row_tab = reinterpret_cast<uint32_t *>(omega_pows + n);
        H2V_CU(cudaMemsetAsync(K.pbits.p, 0, pwords * sizeof(uint32_t), st));
        H2V_CU(cudaMemsetAsync(tmp.first.p, 0xff, cells * sizeof(uint32_t), st));
        H2V_CU(cudaMemsetAsync(row_tab, 0xff, 2 * (size_t)n * sizeof(uint32_t), st));
        // w = GENERATOR^((r - 1) / 2^k), the 2^k-th root of unity EvaluationDomain::new(_, k) uses
        uint32_t e[8];
        for (int i = 0; i < 8; ++i) e[i] = Fr::m(i);
        e[0] -= 1;
        for (int i = 0; i < 8; ++i) e[i] = (e[i] >> K.k) | (i < 7 ? e[i + 1] << (32 - K.k) : 0);
        const fe omega = fe_pow<Fr>(host_fe(7), e);
        mock_omega_table_kernel<<<(n + 255) / 256, 256, 0, st>>>(omega, n, omega_pows, row_tab, 2 * n - 1);
        H2V_LAUNCHED();
        PermKeyArgs pa{};
        pa.sigma = sigma;
        pa.col_vals = reinterpret_cast<const fe *>(tb + ptr_bytes);
        pa.dinv = pa.col_vals + P;
        pa.col_tab = reinterpret_cast<const uint32_t *>(tb + ptr_bytes + fe_bytes);
        pa.omega_pows = omega_pows;
        pa.row_tab = row_tab;
        pa.col_mask = col_slots - 1;
        pa.row_mask = 2 * n - 1;
        pa.k = K.k;
        pa.n = n;
        pa.u = K.u;
        pa.img = K.img.as<uint32_t>();
        pa.first = tmp.first.as<uint32_t>();
        pa.bits = K.pbits.as<uint32_t>();
        mock_perm_decode_kernel<<<dim3((n + 255) / 256, P), 256, 0, st>>>(pa);
        H2V_LAUNCHED();
        mock_perm_key_kernel<<<dim3((n + 255) / 256, P), 256, 0, st>>>(pa);
        H2V_LAUNCHED();
    }
    H2V_CU(cudaStreamSynchronize(st));
    *out = key.release();
    return H2V_OK;
}

size_t mock_witness_bytes(const MockKey &K) {
    const size_t groups = K.wbits / (32 * GROUP_WORDS);
    return ((size_t)K.A + K.I) * K.n * sizeof(fe) + K.wbits / 8 + 3 * groups * sizeof(uint32_t) + 4096;
}
size_t mock_max_batch(const MockKey &K) {
    // every flag index of a batch, and so every compaction offset, fits in 32 bits; witnesses go on grid.z
    return std::max<size_t>(1, std::min<size_t>(65535, (((uint64_t)1 << 32) - 1) / std::max<uint64_t>(K.wbits, 1)));
}

int mock_stage(cudaStream_t st, const MockKey &K, size_t B, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
               const uint32_t *const *instance_len, DevBuf &adv, DevBuf &inst, double ms[2]) {
    const uint32_t n = K.n, A = K.A, I = K.I;
    const double t0 = now_ms();
    H2V_TRY(adv.ensure(B * A * n * sizeof(fe)));
    H2V_TRY(inst.ensure(std::max<size_t>(1, B * I) * n * sizeof(fe)));
    fe *adv_d = adv.as<fe>(), *inst_d = inst.as<fe>();
    for (size_t w = 0; w < B; ++w)
        for (uint32_t c = 0; c < A; ++c)
            H2V_CU(cudaMemcpyAsync(adv_d + (w * A + c) * n, advice[w][c], n * sizeof(fe), cudaMemcpyHostToDevice, st));
    if (I) H2V_CU(cudaMemsetAsync(inst_d, 0, B * I * n * sizeof(fe), st));
    for (size_t w = 0; w < B; ++w)
        for (uint32_t c = 0; c < I; ++c)
            if (instance_len[w][c])
                H2V_CU(cudaMemcpyAsync(inst_d + (w * I + c) * n, instances[w][c], instance_len[w][c] * sizeof(fe), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaStreamSynchronize(st));
    ms[0] += now_ms() - t0;
    return H2V_OK;
}

int mock_check(cudaStream_t st, const MockKey &K, size_t B, const fe *adv_d, const fe *inst_d, h2v_mock_failure_t *failures_out, size_t cap,
               uint64_t *n_failures, double ms[2]) {
    const uint32_t n = K.n, A = K.A, I = K.I;
    const double t1 = now_ms();

    // flags: every witness's section zeroed, the key's permutation flags copied in
    struct Scratch {
        DevBuf bits, scan, out;
        ~Scratch() {
            for (DevBuf *b : {&bits, &scan, &out}) b->release();
        }
    } m;
    const uint64_t wwords = K.wbits / 32, n_words = B * wwords;
    const uint32_t gpw = (uint32_t)(wwords / GROUP_WORDS), n_groups = (uint32_t)(B * gpw), n_tiles = (n_groups + 2047) / 2048;
    std::vector<uint32_t> firsts(B + 1, 0);
    if (n_groups) {
        H2V_TRY(m.bits.ensure(n_words * sizeof(uint32_t)));
        H2V_TRY(m.scan.ensure(((size_t)3 * n_groups + n_tiles + 1) * sizeof(uint32_t)));
        uint32_t *bits = m.bits.as<uint32_t>(), *counts = m.scan.as<uint32_t>(), *offs = counts + n_groups, *scratch = offs + n_groups;
        uint32_t *tiles = scratch + n_groups, *total = tiles + n_tiles;
        H2V_CU(cudaMemsetAsync(bits, 0, n_words * sizeof(uint32_t), st));
        const size_t pwords = (4ull * K.P * n + 31) / 32;
        if (K.P)
            for (size_t w = 0; w < B; ++w)
                H2V_CU(cudaMemcpyAsync(bits + w * wwords + K.perm_base / 32, K.pbits.p, pwords * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        const Batch b{adv_d, inst_d, K.fixed, A, I, K.k, n, K.u, K.wbits, bits};
        if (K.G) {
            mock_gate_kernel<<<dim3((n + 255) / 256, K.G, (unsigned)B), 256, 0, st>>>(b, K.sel(), K.gadv());
            H2V_LAUNCHED();
        }
        if (K.L) {
            mock_lookup_kernel<<<dim3((K.u + 255) / 256, K.L, (unsigned)B), 256, 0, st>>>(b, K.lin(), K.keys.as<fe>(), K.tmap(), K.n_pad, K.lookup_base);
            H2V_LAUNCHED();
        }
        if (K.P) {
            mock_copy_kernel<<<dim3((n + 255) / 256, K.P, (unsigned)B), 256, 0, st>>>(b, K.img.as<uint32_t>(), K.pkind(), K.pidx(), K.perm_base);
            H2V_LAUNCHED();
        }
        mock_count_kernel<<<(n_groups + 255) / 256, 256, 0, st>>>(bits, n_groups, counts);
        H2V_LAUNCHED();
        H2V_TRY(scan_u32_dev(st, counts, n_groups, offs, tiles, scratch, total));
        // the first offset of every witness, and the total
        H2V_CU(cudaMemcpy2DAsync(firsts.data(), sizeof(uint32_t), offs, (size_t)gpw * sizeof(uint32_t), sizeof(uint32_t), B, cudaMemcpyDeviceToHost, st));
        H2V_CU(cudaMemcpyAsync(firsts.data() + B, total, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        H2V_CU(cudaStreamSynchronize(st));
        uint32_t n_out = 0;      // the most failures one witness writes
        for (size_t w = 0; w < B; ++w) n_out = (uint32_t)std::max<uint64_t>(n_out, std::min<uint64_t>(cap, firsts[w + 1] - firsts[w]));
        if (n_out) {
            H2V_TRY(m.out.ensure(B * n_out * sizeof(h2v_mock_failure_t)));
            const Sections s{K.k, n, K.u, gpw, K.lookup_base, K.perm_base, K.gadv(), K.lin(), K.img.as<uint32_t>()};
            mock_emit_kernel<<<(n_groups + 255) / 256, 256, 0, st>>>(bits, n_groups, offs, n_out, s, m.out.as<h2v_mock_failure_t>());
            H2V_LAUNCHED();
            for (size_t w = 0; w < B; ++w) {
                const size_t got = std::min<uint64_t>(cap, firsts[w + 1] - firsts[w]);
                if (got)
                    H2V_CU(cudaMemcpyAsync(failures_out + w * cap, m.out.as<h2v_mock_failure_t>() + w * n_out, got * sizeof(h2v_mock_failure_t),
                                           cudaMemcpyDeviceToHost, st));
            }
        }
        H2V_CU(cudaStreamSynchronize(st));
    }
    for (size_t w = 0; w < B; ++w) n_failures[w] = firsts[w + 1] - firsts[w];
    ms[1] += now_ms() - t1;
    return H2V_OK;
}

void mock_set_last_ms(const double ms[2]) {
    t_last_ms[0] = ms[0];
    t_last_ms[1] = ms[1];
}

// The argument checks of both entry points (who: the prefix of the error text)
int mock_check_advice(const h2v_circuit_t *cs, const uint64_t *const *advice, const char *who) {
    for (uint32_t c = 0; c < cs->n_advice; ++c)
        if (!advice[c]) return failf(H2V_EINVAL, "%s: advice column %u is NULL", who, c);
    return H2V_OK;
}
int mock_check_instances(const h2v_circuit_t *cs, const uint64_t *const *instances, const uint32_t *instance_len, const char *who) {
    const size_t n = (size_t)1 << cs->k;
    for (uint32_t c = 0; c < cs->n_instance; ++c) {
        if (instance_len[c] > n) return failf(H2V_EINVAL, "%s: instance column %u has %u values, more than 2^k = %zu", who, c, instance_len[c], n);
        if (instance_len[c] && !instances[c]) return failf(H2V_EINVAL, "%s: instance column %u is NULL", who, c);
    }
    return H2V_OK;
}
int mock_check_limits(const h2v_circuit_t *cs, const char *who) {
    const uint64_t n = (uint64_t)1 << cs->k, flags = ((uint64_t)cs->n_gates + cs->n_lookups + 4ull * cs->n_perm) * n;
    if (cs->n_gates > 65535 || cs->n_lookups > 65535 || cs->n_perm > 65535)
        return failf(H2V_EINVAL, "%s: more than 65535 gates, lookups or permutation columns", who);
    if (flags >= (1ull << 32))
        return failf(H2V_EINVAL, "%s: (gates + lookups + 4 permutation columns) x 2^k = %llu flags, more than 2^32", who, (unsigned long long)flags);
    return H2V_OK;
}

}  // namespace h2v

namespace {

// h2v_mock_prover: the fixed and sigma columns uploaded, the key tables built from them, a check of one witness
int mock_run(const h2v_circuit_t *cs, const uint64_t *const *fixed, const uint64_t *const *sigma, const uint64_t *const *advice,
             const uint64_t *const *instances, const uint32_t *instance_len, h2v_mock_failure_t *failures_out, size_t cap,
             uint64_t *n_failures) {
    const size_t n = (size_t)1 << cs->k;
    const uint32_t F = cs->n_fixed, P = cs->n_perm;
    struct Call {
        DevBuf cols, adv, inst;
        MockKey *key = nullptr;
        cudaStream_t st = nullptr;
        ~Call() {
            mock_key_free(key);
            for (DevBuf *b : {&cols, &adv, &inst}) b->release();
            if (st) cudaStreamDestroy(st);
        }
    } m;
    H2V_CU(cudaStreamCreateWithFlags(&m.st, cudaStreamNonBlocking));
    const double t0 = now_ms();
    H2V_TRY(m.cols.ensure(std::max<size_t>((size_t)F + P, 1) * n * sizeof(fe)));
    fe *fix_d = m.cols.as<fe>(), *sig_d = fix_d + (size_t)F * n;
    for (uint32_t c = 0; c < F; ++c) H2V_CU(cudaMemcpyAsync(fix_d + (size_t)c * n, fixed[c], n * sizeof(fe), cudaMemcpyHostToDevice, m.st));
    for (uint32_t c = 0; c < P; ++c) H2V_CU(cudaMemcpyAsync(sig_d + (size_t)c * n, sigma[c], n * sizeof(fe), cudaMemcpyHostToDevice, m.st));
    H2V_CU(cudaStreamSynchronize(m.st));
    const double t1 = now_ms();
    H2V_TRY(mock_key_build(m.st, cs, fix_d, sig_d, &m.key));
    double ms[2] = {t1 - t0, now_ms() - t1};
    H2V_TRY(mock_stage(m.st, *m.key, 1, &advice, &instances, &instance_len, m.adv, m.inst, ms));
    H2V_TRY(mock_check(m.st, *m.key, 1, m.adv.as<fe>(), m.inst.as<fe>(), failures_out, cap, n_failures, ms));
    mock_set_last_ms(ms);
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
    H2V_TRY(mock_check_advice(cs, advice, "mock_prover"));
    for (uint32_t c = 0; c < cs->n_fixed; ++c)
        if (!fixed[c]) return failf(H2V_EINVAL, "mock_prover: fixed column %u is NULL", c);
    for (uint32_t c = 0; c < cs->n_perm; ++c)
        if (!sigma[c]) return failf(H2V_EINVAL, "mock_prover: sigma column %u is NULL", c);
    H2V_TRY(mock_check_instances(cs, instances, instance_len, "mock_prover"));
    H2V_TRY(mock_check_limits(cs, "mock_prover"));
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
