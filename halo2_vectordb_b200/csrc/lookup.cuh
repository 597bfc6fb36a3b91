// lookup.cuh -- the lookup argument's permuted columns A', S' (create_proof step 5, SURVEY.md 3.1).
//
// Replaces halo2-axiom plonk/lookup/prover.rs `permute_expression_pair` [UPSTREAM; reached from
// /root/reference/src/scaffold/mod.rs:296]: A' = the first `usable_rows` input values sorted (Ord on Fr = order of the
// canonical integers); S' carries A'[i] on every row where A' changes, and the table values that are left over
// (table multiset minus one copy of every distinct input value), ascending, on the remaining rows taken from the LAST
// repeated row backwards (upstream pops `repeated_input_rows` from the end).  An input value missing from the table is
// an error (upstream: Error::ConstraintSystemFailure).
//
// Device plan (byte / index work, L2-resident at prover sizes): canonicalise + pad to a power of two with all-ones
// keys, bitonic sort of the 256-bit keys (shared-memory kernels below 1024-element strides, one global pass per larger
// stride), first-occurrence flags + binary search into the sorted table, two exclusive scans, two scatters.
#pragma once
#include "ff.cuh"

namespace h2v {

typedef FrP FrL;
#define H2V_SORT_TILE 1024u          // elements per shared-memory tile (32 KiB)


// out[i] = canonical(in[i]) for i < n, all-ones (greater than any field element) for n <= i < n_pad
// (grid.y = 0: input -> keys[0 .. n_pad), grid.y = 1: table -> keys[n_pad .. 2 n_pad): both sorts share every launch)
__global__ void lookup_canon_pad_kernel(const fe *__restrict__ in0, const fe *__restrict__ in1, fe *__restrict__ out, uint32_t n,
                                        uint32_t n_pad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    const fe *in = blockIdx.y ? in1 : in0;
    out += (size_t)blockIdx.y * n_pad;
    fe r;
    if (i < n) {
        r = fe_from_mont<FrL>(fe_load_global(in + i));
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) r.v[k] = 0xffffffffu;
    }
    fe_store_global(out + i, r);
}

// compare-exchange of the pair (i, i + j) inside the bitonic block of size k
__device__ __forceinline__ void bitonic_cx(fe &lo, fe &hi, bool ascending) {
    if (key_less(hi, lo) == ascending) {
        fe t = lo;
        lo = hi;
        hi = t;
    }
}
// one (k, j) step with j >= H2V_SORT_TILE: one thread per pair, straight from global memory
__global__ void __launch_bounds__(256) bitonic_global_kernel(fe *__restrict__ a, uint32_t n_pad, uint32_t k, uint32_t j) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pad / 2) return;
    a += (size_t)blockIdx.y * n_pad;
    uint32_t i = 2 * j * (p / j) + (p % j);
    fe x = fe_load_global(a + i), y = fe_load_global(a + i + j);
    bitonic_cx(x, y, (i & k) == 0);
    fe_store_global(a + i, x);
    fe_store_global(a + i + j, y);
}
// all steps of one tile that stay inside it: either the complete sort of the tile (k = 2 .. tile, full == 1) or the
// tail j = tile/2 .. 1 of a larger k.  blockDim = tile / 2.
__global__ void __launch_bounds__(H2V_SORT_TILE / 2) bitonic_tile_kernel(fe *__restrict__ a, uint32_t n_pad, uint32_t k_outer, int full) {
    extern __shared__ uint4 sort_smem[];
    fe *s = reinterpret_cast<fe *>(sort_smem);
    const uint32_t tile = min(H2V_SORT_TILE, n_pad);
    const uint32_t base = blockIdx.x * tile;
    const uint32_t t = threadIdx.x;
    a += (size_t)blockIdx.y * n_pad;
    if (t < tile / 2) {
        s[t] = fe_load_global(a + base + t);
        s[t + tile / 2] = fe_load_global(a + base + t + tile / 2);
    }
    __syncthreads();
    for (uint32_t k = full ? 2 : k_outer; k <= (full ? tile : k_outer); k <<= 1) {
        for (uint32_t j = min(k >> 1, tile >> 1); j > 0; j >>= 1) {
            if (t < tile / 2) {
                uint32_t i = 2 * j * (t / j) + (t % j);
                fe x = s[i], y = s[i + j];
                bitonic_cx(x, y, ((base + i) & k) == 0);
                s[i] = x;
                s[i + j] = y;
            }
            __syncthreads();
        }
    }
    if (t < tile / 2) {
        fe_store_global(a + base + t, s[t]);
        fe_store_global(a + base + t + tile / 2, s[t + tile / 2]);
    }
}

__global__ void lookup_fill_kernel(uint32_t *a, uint32_t v, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}
// rep[i] = 1 when sorted input row i repeats row i-1; for a first occurrence, the first table entry with the same
// value is taken out of the leftover set (free[pos] = 0); a value missing from the table raises *err
__global__ void lookup_flags_kernel(const fe *__restrict__ As, const fe *__restrict__ Ts, uint32_t u, uint32_t *__restrict__ rep,
                                    uint32_t *__restrict__ free_, int *__restrict__ err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= u) return;
    fe v = fe_load_global(As + i);
    bool first = i == 0 || !key_eq(v, fe_load_global(As + i - 1));
    rep[i] = first ? 0u : 1u;
    if (!first) return;
    uint32_t lo = 0, hi = u;      // lower bound of v in Ts[0 .. u)
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (key_less(fe_load_global(Ts + mid), v)) lo = mid + 1;
        else hi = mid;
    }
    if (lo < u && key_eq(fe_load_global(Ts + lo), v)) free_[lo] = 0u;
    else atomicExch(err, 1);
}
// rep_rows[r] = the r-th repeated row; A' and the first-occurrence rows of S' are written in Montgomery form
__global__ void lookup_emit_input_kernel(const fe *__restrict__ As, uint32_t u, const uint32_t *__restrict__ rep,
                                         const uint32_t *__restrict__ rep_offs, uint32_t *__restrict__ rep_rows, fe *__restrict__ out_a,
                                         fe *__restrict__ out_s) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= u) return;
    fe m = fe_to_mont<FrL>(fe_load_global(As + i));
    fe_store_global(out_a + i, m);
    if (rep[i]) rep_rows[rep_offs[i]] = i;
    else fe_store_global(out_s + i, m);
}
// the k-th leftover table value (ascending) goes to the (m - 1 - k)-th repeated row
__global__ void lookup_emit_table_kernel(const fe *__restrict__ Ts, uint32_t u, const uint32_t *__restrict__ free_,
                                         const uint32_t *__restrict__ free_offs, const uint32_t *__restrict__ totals,
                                         const uint32_t *__restrict__ rep_rows, fe *__restrict__ out_s, int *__restrict__ err) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= u || !free_[p]) return;
    const uint32_t m = totals[0];            // number of repeated rows
    if (totals[1] != m) {                    // cannot happen when every input value was found; defensive
        atomicCAS(err, 0, 2);      // keep an earlier "missing value" report
        return;
    }
    uint32_t row = rep_rows[m - 1 - free_offs[p]];
    fe_store_global(out_s + row, fe_to_mont<FrL>(fe_load_global(Ts + p)));
}

// ---- the same plan for ALL lookup arguments of a proof in one set of launches (a kmeans-sized proof has 72 of them over
// one shared table: one at a time they are 72 x ~35 launches of 32-block grids).  keys[y][0 .. n_pad): slice y < L holds the
// sorted input of lookup y, slice L + t the sorted t-th DISTINCT table; tmap[l] = the table slice of lookup l.  The
// per-lookup index arrays are rows of [L][u] matrices scanned as one long array; a row's own offsets are the scanned
// values minus the value at the row's start.
__global__ void lookup_canon_pad_batch_kernel(const fe *const *__restrict__ srcs, fe *__restrict__ out, uint32_t n, uint32_t n_pad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    const fe *in = srcs[blockIdx.y];
    out += (size_t)blockIdx.y * n_pad;
    fe r;
    if (i < n) {
        r = fe_from_mont<FrL>(fe_load_global(in + i));
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) r.v[k] = 0xffffffffu;
    }
    fe_store_global(out + i, r);
}
__global__ void lookup_flags_batch_kernel(const fe *__restrict__ keys, const uint32_t *__restrict__ tmap, uint32_t u, uint32_t n_pad,
                                          uint32_t *__restrict__ rep, uint32_t *__restrict__ free_, int *__restrict__ err) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= u) return;
    const uint32_t l = blockIdx.y;
    const fe *As = keys + (size_t)l * n_pad, *Ts = keys + (size_t)tmap[l] * n_pad;
    rep += (size_t)l * u;
    free_ += (size_t)l * u;
    fe v = fe_load_global(As + i);
    bool first = i == 0 || !key_eq(v, fe_load_global(As + i - 1));
    rep[i] = first ? 0u : 1u;
    if (!first) return;
    uint32_t lo = 0, hi = u;      // lower bound of v in Ts[0 .. u)
    while (lo < hi) {
        uint32_t mid = (lo + hi) >> 1;
        if (key_less(fe_load_global(Ts + mid), v)) lo = mid + 1;
        else hi = mid;
    }
    if (lo < u && key_eq(fe_load_global(Ts + lo), v)) free_[lo] = 0u;
    else atomicExch(err, 1);
}
__global__ void lookup_emit_input_batch_kernel(const fe *__restrict__ keys, uint32_t u, uint32_t n_pad, const uint32_t *__restrict__ rep,
                                               const uint32_t *__restrict__ rep_offs, uint32_t *__restrict__ rep_rows,
                                               fe *__restrict__ out_a, size_t a_stride, fe *__restrict__ out_s, size_t s_stride) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= u) return;
    const uint32_t l = blockIdx.y;
    const size_t row0 = (size_t)l * u;
    fe m = fe_to_mont<FrL>(fe_load_global(keys + (size_t)l * n_pad + i));
    fe_store_global(out_a + l * a_stride + i, m);
    if (rep[row0 + i]) rep_rows[row0 + (rep_offs[row0 + i] - rep_offs[row0])] = i;
    else fe_store_global(out_s + l * s_stride + i, m);
}
__global__ void lookup_emit_table_batch_kernel(const fe *__restrict__ keys, const uint32_t *__restrict__ tmap, uint32_t n_lookups, uint32_t u,
                                               uint32_t n_pad, const uint32_t *__restrict__ free_, const uint32_t *__restrict__ free_offs,
                                               const uint32_t *__restrict__ rep_offs, const uint32_t *__restrict__ totals,
                                               const uint32_t *__restrict__ rep_rows, fe *__restrict__ out_s, size_t s_stride,
                                               int *__restrict__ err) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t l = blockIdx.y;
    const size_t row0 = (size_t)l * u;
    if (p >= u || !free_[row0 + p]) return;
    const bool last = l + 1 == n_lookups;
    const uint32_t m = (last ? totals[0] : rep_offs[row0 + u]) - rep_offs[row0];            // repeated rows of this lookup
    const uint32_t mf = (last ? totals[1] : free_offs[row0 + u]) - free_offs[row0];          // leftover table values
    if (mf != m) {                    // cannot happen when every input value was found; defensive
        atomicCAS(err, 0, 2);         // keep an earlier "missing value" report
        return;
    }
    uint32_t row = rep_rows[row0 + (m - 1 - (free_offs[row0 + p] - free_offs[row0]))];
    fe_store_global(out_s + l * s_stride + row, fe_to_mont<FrL>(fe_load_global(keys + (size_t)tmap[l] * n_pad + p)));
}

}  // namespace h2v
