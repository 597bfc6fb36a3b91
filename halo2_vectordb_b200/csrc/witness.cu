// witness.cu -- witness generation on the device: a recorded circuit (circuit.cu: make_plan) replayed for a batch of
// inputs, then gathered into the advice columns and instances h2v_builder_layout would give for each input.
//
// One cooperative kernel evaluates the program level by level over (witness, cell) pairs, with a grid-wide barrier
// between levels (a program has 10^3 - 10^5 levels: one launch per level would cost more than the work).  Values are
// canonical, as the host builder keeps them, so that the integer rules (bits, limbs, division, MSB, low-32 compares) read
// the same integers; field products are Montgomery products followed by a multiplication by R^2.  A second kernel writes
// the Montgomery-form columns.
#include <cooperative_groups.h>

#include <algorithm>
#include <chrono>
#include <mutex>

#include "ff.cuh"
#include "internal.hpp"
#include "zk_builder.hpp"

using namespace h2v;
namespace cg = cooperative_groups;

struct h2v_witness_program {
    WitnessPlan plan;      // rules, pool and map move to the device on the first h2v_witness_generate
    std::mutex mu;
    bool uploaded = false;
    int dev = 0, grid = 0;
    uint64_t n_computed = 0, n_pool = 0, n_map = 0;
    DevBuf rules, cell_of, level_start, pool, map;      // the program
    DevBuf in, vals, adv, inst, err;                   // one group of witnesses
    size_t witness_bytes() const {
        return sizeof(fe) * (plan.n_inputs * 2 + n_computed + plan.n_adv_cols * ((size_t)1 << plan.k) + plan.n_instances) + 8;
    }
};

namespace {

constexpr int WG_THREADS = 256;
enum : uint32_t { WERR_DIV_ZERO = 1, WERR_POW2_INDEX = 2 };
const char *werr_text(uint32_t code) {
    return code == WERR_DIV_ZERO ? "attempt to divide by zero" : code == WERR_POW2_INDEX ? "index out of bounds: pow_of_two" : "unknown error";
}
double t_last_ms[3] = {0, 0, 0};

__device__ __forceinline__ fe fr_mul(const fe &a, const fe &b) { return fe_to_mont<FrP>(fe_mul<FrP>(a, b)); }      // (ab/R) R^2 / R
__device__ __forceinline__ fe small(uint32_t x) {
    fe r = fe_zero();
    r.v[0] = x;
    return r;
}
__device__ __forceinline__ fe pow2(uint32_t i) {      // 2^i, i < 256
    fe r = fe_zero();
    r.v[i >> 5] = 1u << (i & 31);
    return r;
}
// (a >> shift) mod 2^width, shift < 256, width <= 256
__device__ __forceinline__ fe bits(const fe &a, uint32_t shift, uint32_t width) {
    fe r;
    const uint32_t w = shift >> 5, b = shift & 31;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t lo = i + w < 8 ? a.v[i + w] : 0u, hi = i + w + 1 < 8 ? a.v[i + w + 1] : 0u;
        r.v[i] = b ? (lo >> b) | (hi << (32 - b)) : lo;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int keep = (int)width - 32 * i;
        r.v[i] = keep >= 32 ? r.v[i] : keep <= 0 ? 0u : r.v[i] & ((1u << keep) - 1u);
    }
    return r;
}
__device__ __forceinline__ int top_bit(const fe &a) {      // index of the highest set bit, -1 for 0
    for (int i = 7; i >= 0; --i)
        if (a.v[i]) return 32 * i + 31 - __clz(a.v[i]);
    return -1;
}
__device__ __forceinline__ bool less(const fe &a, const fe &b) {
    fe d;
    return raw_sub(d.v, a.v, b.v) != 0;
}
// BigUint floor division, as zk_builder.hpp's u_divmod (b != 0)
__device__ __noinline__ void divmod(const fe &a, const fe &b, fe &q, fe &r) {
    q = fe_zero();
    r = fe_zero();
    for (int i = top_bit(a); i >= 0; --i) {
#pragma unroll
        for (int j = 7; j > 0; --j) r.v[j] = (r.v[j] << 1) | (r.v[j - 1] >> 31);
        r.v[0] = (r.v[0] << 1) | ((a.v[i >> 5] >> (i & 31)) & 1u);
        fe d;
        if (!raw_sub(d.v, r.v, b.v)) {
            r = d;
            q.v[i >> 5] |= 1u << (i & 31);
        }
    }
}
__device__ __noinline__ fe inv_or_one(const fe &a) {
    if (fe_is_zero(a)) return small(1);
    return fe_from_mont<FrP>(fe_inv_fast<FrP>(fe_to_mont<FrP>(a)));
}
__device__ __forceinline__ fe modulus() {
    fe m;
#pragma unroll
    for (int i = 0; i < 8; ++i) m.v[i] = FrP::m(i);
    return m;
}
// signed_div_scale (zk_chips.hpp) for the divisor 2^p: q (want_q) or r
__device__ __noinline__ fe signed_div_scale(const fe &a, uint32_t p, bool want_q) {
    const fe m = modulus();
    if (!less(pow2(252), a)) return want_q ? bits(a, p, 256) : bits(a, 0, p);
    fe a_abs, dq, q, prod, r;
    raw_sub(a_abs.v, m.v, a.v);      // r - a
    dq = bits(a_abs, p, 256);
    if (!fe_is_zero(bits(a_abs, 0, p))) {
        const fe one = small(1);
        raw_add(dq.v, dq.v, one.v);
    }
    raw_sub(q.v, m.v, dq.v);         // r - ceil(|a| / 2^p)
    if (want_q) return q;
    prod = fr_mul(pow2(p), q);
    raw_sub(r.v, a.v, prod.v);       // wrapping, then one conditional subtraction of r (f_from_u)
    fe d;
    if (!raw_sub(d.v, r.v, m.v)) r = d;
    return r;
}
// quantization((double)low128(a)) at precision p (hamming_distance's count)
__device__ __noinline__ fe qcount(const fe &a, uint32_t p) {
    const uint64_t lo = ((uint64_t)a.v[1] << 32) | a.v[0], hi = ((uint64_t)a.v[3] << 32) | a.v[2];
    double d;
    if (!hi) {
        d = __ull2double_rn(lo);
    } else {      // correctly rounded: the top 64 bits with the rest folded into a sticky bit
        const int s = __clzll((long long)hi);
        uint64_t top = s ? (hi << s) | (lo >> (64 - s)) : hi;
        if (lo << s) top |= 1;
        d = ldexp(__ull2double_rn(top), 64 - s);
    }
    const double scaled = d * ldexp(1.0, (int)p);      // exact: d is an integer below 2^128, round() leaves it as is
    fe r = fe_zero();
    if (!(scaled > 0)) return r;
    if (scaled >= 340282366920938463463374607431768211456.0) {      // Rust `as u128` saturates
#pragma unroll
        for (int i = 0; i < 4; ++i) r.v[i] = 0xffffffffu;
        return r;
    }
    const uint64_t bits_ = (uint64_t)__double_as_longlong(scaled);
    const int e = (int)((bits_ >> 52) & 0x7ff) - 1075;      // scaled = m 2^e
    const uint64_t mant = (bits_ & ((1ull << 52) - 1)) | (1ull << 52);
    uint64_t o[2] = {0, 0};
    if (e < 0) {
        o[0] = mant >> -e;
    } else if (e < 64) {
        o[0] = mant << e;
        o[1] = e ? mant >> (64 - e) : 0;
    } else {
        o[1] = mant << (e - 64);
    }
    r.v[0] = (uint32_t)o[0];
    r.v[1] = (uint32_t)(o[0] >> 32);
    r.v[2] = (uint32_t)o[1];
    r.v[3] = (uint32_t)(o[1] >> 32);
    return r;
}
__device__ __forceinline__ uint32_t msb_index(const fe &a) {      // qlog2's num_digits: 1 when a == 0
    const int t = top_bit(a);
    return t < 0 ? 1u : (uint32_t)t;
}

__device__ __forceinline__ fe load(uint32_t ref, const fe *vals, const fe *pool) {
    if (ref == WREF_ZERO) return fe_zero();
    return (ref & WREF_POOL) ? pool[ref & ~WREF_POOL] : vals[ref];
}

__device__ __forceinline__ fe eval(const WitnessRule &r, const fe *vals, const fe *pool, uint32_t &err) {
    const uint32_t kind = r.op & 255, imm = r.op >> 8;
    const fe a = load(r.a, vals, pool);
    switch (kind) {
        case zk::OP_ADD: return fe_add<FrP>(a, load(r.b, vals, pool));
        case zk::OP_SUB: return fe_sub<FrP>(a, load(r.b, vals, pool));
        case zk::OP_NEG: return fe_neg<FrP>(a);
        case zk::OP_MUL: return fr_mul(a, load(r.b, vals, pool));
        case zk::OP_MUL_ADD: return fe_add<FrP>(fr_mul(a, load(r.b, vals, pool)), load(r.c, vals, pool));
        case zk::OP_OR: {
            const fe b = load(r.b, vals, pool);
            return fe_sub<FrP>(fe_add<FrP>(a, b), fr_mul(a, b));
        }
        case zk::OP_IS_ZERO: return small(fe_is_zero(a) ? 1u : 0u);
        case zk::OP_INV_OR_ONE: return inv_or_one(a);
        case zk::OP_BITS: return bits(a, imm & 255, imm >> 8);
        case zk::OP_DIV_Q:
        case zk::OP_DIV_R: {
            const fe b = load(r.b, vals, pool);
            if (fe_is_zero(b)) {
                err = WERR_DIV_ZERO;
                return fe_zero();
            }
            fe q, rem;
            divmod(a, b, q, rem);
            return kind == zk::OP_DIV_Q ? q : rem;
        }
        case zk::OP_SDS_Q: return signed_div_scale(a, imm, true);
        case zk::OP_SDS_R: return signed_div_scale(a, imm, false);
        case zk::OP_IND: return small(a.v[0] == imm ? 1u : 0u);
        case zk::OP_IND_VAL: return a.v[0] == imm ? a : fe_zero();
        case zk::OP_SELECT_IND: return fe_is_zero(load(r.b, vals, pool)) ? load(r.c, vals, pool) : a;
        case zk::OP_MSB: return small(msb_index(a));
        case zk::OP_POW2_MSB:
        case zk::OP_POW2_LOW32: {
            const uint32_t i = kind == zk::OP_POW2_MSB ? msb_index(a) : a.v[0];
            if (i >= 254) {
                err = WERR_POW2_INDEX;
                return fe_zero();
            }
            return pow2(i);
        }
        case zk::OP_QCOUNT: return qcount(a, imm);
    }
    return fe_zero();
}

// B witnesses: vals + w S holds witness w's inputs (slots [0, n_inputs)) then its computed cells.  err[w] = the least
// (trace cell << 8 | code) of the witness's failing cells.
__global__ void __launch_bounds__(WG_THREADS) witness_eval(const WitnessRule *__restrict__ rules, const uint32_t *__restrict__ cell_of,
                                                           const uint32_t *__restrict__ level_start, uint32_t n_levels,
                                                           const fe *__restrict__ pool, const fe *__restrict__ in, fe *vals, uint64_t S,
                                                           uint32_t n_inputs, uint32_t B, unsigned long long *err) {
    cg::grid_group grid = cg::this_grid();
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x, t0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (uint64_t t = t0; t < (uint64_t)B * n_inputs; t += stride) {
        const uint64_t w = t / n_inputs;
        vals[w * S + (t - w * n_inputs)] = fe_from_mont<FrP>(in[t]);
    }
    grid.sync();
    uint32_t c0 = level_start[0];
    for (uint32_t l = 1; l <= n_levels; ++l) {      // level l: rules [level_start[l - 1], level_start[l])
        const uint32_t c1 = level_start[l], cnt = c1 - c0;
        for (uint64_t t = t0; t < (uint64_t)B * cnt; t += stride) {
            const uint64_t w = t / cnt;
            const uint32_t c = c0 + (uint32_t)(t - w * cnt);
            fe *vw = vals + w * S;
            uint32_t e = 0;
            const fe v = eval(rules[c], vw, pool, e);
            vw[n_inputs + c] = v;
            if (e) atomicMin(err + w, (unsigned long long)cell_of[c] << 8 | e);
        }
        grid.sync();
        c0 = c1;
    }
}

// adv: B witnesses x (A n advice cells); inst: B x inst_stride, witness w's n_inst instances then zeros (inst_stride >=
// n_inst); Montgomery form
__global__ void __launch_bounds__(WG_THREADS) witness_gather(const uint32_t *__restrict__ map, uint64_t n_adv, uint64_t n_inst,
                                                             uint64_t inst_stride, const fe *__restrict__ pool, const fe *__restrict__ vals,
                                                             uint64_t S, uint32_t B, fe *adv, fe *inst) {
    const uint64_t P = n_adv + inst_stride, stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < (uint64_t)B * P; t += stride) {
        const uint64_t w = t / P, pos = t - w * P;
        const uint32_t ref = pos < n_adv + n_inst ? map[pos] : WREF_ZERO;
        const fe v = ref == WREF_ZERO ? fe_zero() : fe_to_mont<FrP>(load(ref, vals + w * S, pool));
        if (pos < n_adv) adv[w * n_adv + pos] = v;
        else inst[w * inst_stride + (pos - n_adv)] = v;
    }
}

double ms_since(std::chrono::steady_clock::time_point &t) {
    const auto now = std::chrono::steady_clock::now();
    const double ms = std::chrono::duration<double, std::milli>(now - t).count();
    t = now;
    return ms;
}

// the program to the current device, in copies on st
int upload(h2v_witness_program *p, cudaStream_t st) {
    WitnessPlan &P = p->plan;
    p->n_computed = P.rules.size();
    p->n_pool = P.pool.size() / 4;
    p->n_map = P.map.size();
    H2V_TRY(p->rules.ensure(std::max<size_t>(1, P.rules.size()) * sizeof(WitnessRule)));
    H2V_TRY(p->cell_of.ensure(std::max<size_t>(1, P.cell_of.size()) * sizeof(uint32_t)));
    H2V_TRY(p->level_start.ensure(P.level_start.size() * sizeof(uint32_t)));
    H2V_TRY(p->pool.ensure(std::max<size_t>(1, p->n_pool) * sizeof(fe)));
    H2V_TRY(p->map.ensure(std::max<size_t>(1, P.map.size()) * sizeof(uint32_t)));
    std::vector<uint32_t> cell32(P.cell_of.begin(), P.cell_of.end());
    H2V_CU(cudaMemcpyAsync(p->rules.p, P.rules.data(), P.rules.size() * sizeof(WitnessRule), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(p->cell_of.p, cell32.data(), cell32.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(p->level_start.p, P.level_start.data(), P.level_start.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(p->pool.p, P.pool.data(), P.pool.size() * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(p->map.p, P.map.data(), P.map.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaStreamSynchronize(st));      // the host vectors are released below
    int blocks = 0, sms = 0;
    H2V_CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, witness_eval, WG_THREADS, 0));
    H2V_CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, p->dev));
    if (blocks < 1) return failf(H2V_ECUDA, "witness_generate: the evaluation kernel cannot be resident");
    p->grid = blocks * sms;
    std::vector<WitnessRule>().swap(P.rules);
    std::vector<uint64_t>().swap(P.pool);
    std::vector<uint32_t>().swap(P.map);
    p->uploaded = true;
    return H2V_OK;
}

// B witnesses (inputs: B x n_inputs x 4 limbs) evaluated and gathered on st: witness w's advice columns to adv + w A n, its
// instances to inst + w inst_stride, zero-padded.  Then downloaded: the advice to advice_out (unless NULL), the instances
// to instances_out + w n_instances 4 (unless NULL).  *bad_w = the first failing witness of the group, or B when none
int run_group(h2v_witness_program *p, cudaStream_t st, size_t B, const uint64_t *inputs, fe *adv, fe *inst, size_t inst_stride,
              uint64_t *advice_out, uint64_t *instances_out, size_t *bad_w, uint64_t *bad_code, double ms[3]) {
    const WitnessPlan &P = p->plan;
    const size_t n = (size_t)1 << P.k, n_adv = P.n_adv_cols * n, n_in = P.n_inputs, S = n_in + p->n_computed;
    auto t = std::chrono::steady_clock::now();
    if (B * n_in) H2V_CU(cudaMemcpyAsync(p->in.p, inputs, B * n_in * sizeof(fe), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemsetAsync(p->err.p, 0xff, B * sizeof(uint64_t), st));
    H2V_CU(cudaStreamSynchronize(st));
    ms[0] += ms_since(t);
    const WitnessRule *rules = p->rules.as<WitnessRule>();
    const uint32_t *cell_of = p->cell_of.as<uint32_t>(), *level_start = p->level_start.as<uint32_t>();
    const fe *pool = p->pool.as<fe>(), *in = p->in.as<fe>();
    fe *vals = p->vals.as<fe>();
    uint32_t n_levels = P.n_levels, n_inputs = (uint32_t)n_in, Bu = (uint32_t)B;
    uint64_t S64 = S;
    unsigned long long *err = p->err.as<unsigned long long>();
    void *args[] = {&rules, &cell_of, &level_start, &n_levels, &pool, &in, &vals, &S64, &n_inputs, &Bu, &err};
    H2V_CU(cudaLaunchCooperativeKernel((const void *)witness_eval, dim3(p->grid), dim3(WG_THREADS), args, 0, st));
    H2V_LAUNCHED();
    const uint64_t total = (uint64_t)B * (n_adv + inst_stride);
    const unsigned gblocks = (unsigned)std::min<uint64_t>((total + WG_THREADS - 1) / WG_THREADS, (uint64_t)p->grid * 8);
    witness_gather<<<std::max(1u, gblocks), WG_THREADS, 0, st>>>(p->map.as<uint32_t>(), n_adv, P.n_instances, inst_stride, pool, vals, S, Bu,
                                                                 adv, inst);
    H2V_LAUNCHED();
    H2V_CU(cudaStreamSynchronize(st));
    ms[1] += ms_since(t);
    std::vector<uint64_t> err_h(B);
    H2V_CU(cudaMemcpyAsync(err_h.data(), p->err.p, B * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    if (advice_out) H2V_CU(cudaMemcpyAsync(advice_out, adv, B * n_adv * sizeof(fe), cudaMemcpyDeviceToHost, st));
    if (P.n_instances && instances_out)
        H2V_CU(cudaMemcpy2DAsync(instances_out, P.n_instances * sizeof(fe), inst, inst_stride * sizeof(fe), P.n_instances * sizeof(fe), B,
                                 cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    ms[2] += ms_since(t);
    *bad_w = B;
    for (size_t w = 0; w < B; ++w)
        if (err_h[w] != ~0ull) {
            *bad_w = w;
            *bad_code = err_h[w];
            break;
        }
    return H2V_OK;
}

// the evaluation buffers of a group of B witnesses
int ensure_eval(h2v_witness_program *p, size_t B) {
    const size_t S = p->plan.n_inputs + p->n_computed;
    H2V_TRY(p->in.ensure(std::max<size_t>(1, B * p->plan.n_inputs) * sizeof(fe)));
    H2V_TRY(p->vals.ensure(std::max<size_t>(1, B * S) * sizeof(fe)));
    return p->err.ensure(B * sizeof(uint64_t));
}

int generate(h2v_witness_program *p, size_t n_witnesses, const uint64_t *inputs, uint64_t *advice_out, uint64_t *instances_out) {
    if (!p->uploaded) H2V_TRY(upload(p, 0));
    const WitnessPlan &P = p->plan;
    const size_t n = (size_t)1 << P.k, n_adv = P.n_adv_cols * n;
    const size_t held = p->in.cap + p->vals.cap + p->adv.cap + p->inst.cap + p->err.cap;
    size_t G = group_size_free(n_witnesses, p->witness_bytes(), 65535, held);
    double ms[3] = {0, 0, 0};
    for (size_t w0 = 0; w0 < n_witnesses;) {
        const size_t B = std::min(G, n_witnesses - w0);
        int rc = ensure_eval(p, B);
        if (!rc) rc = p->adv.ensure(std::max<size_t>(1, B * n_adv) * sizeof(fe));
        if (!rc) rc = p->inst.ensure(std::max<size_t>(1, B * P.n_instances) * sizeof(fe));
        if (rc == H2V_ENOMEM && G > 1) {      // halve the group and try again
            for (DevBuf *b : {&p->in, &p->vals, &p->adv, &p->inst, &p->err}) b->release();
            G = std::max<size_t>(1, G / 2);
            continue;
        }
        H2V_TRY(rc);
        size_t bad = B;
        uint64_t code = 0;
        H2V_TRY(run_group(p, 0, B, inputs + w0 * P.n_inputs * 4, p->adv.as<fe>(), p->inst.as<fe>(), P.n_instances, advice_out + w0 * n_adv * 4,
                          P.n_instances ? instances_out + w0 * P.n_instances * 4 : nullptr, &bad, &code, ms));
        if (bad < B) {
            std::copy(ms, ms + 3, t_last_ms);
            return failf(H2V_EINVAL, "witness_generate: witness %zu: %s (cell %llu)", w0 + bad, werr_text((uint32_t)(code & 255)),
                         (unsigned long long)(code >> 8));
        }
        w0 += B;
    }
    std::copy(ms, ms + 3, t_last_ms);
    return H2V_OK;
}

}  // namespace

namespace h2v {
bool fr_reduced(const uint64_t *x) {
    static const uint64_t M[4] = {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull};
    for (int i = 3; i >= 0; --i)
        if (x[i] != M[i]) return x[i] < M[i];
    return false;
}
std::mutex &witness_program_mutex(h2v_witness_program *p) { return p->mu; }
int witness_program_bind(h2v_witness_program *p, int dev, cudaStream_t st, const char *who, size_t *held) {
    if (p->uploaded && p->dev != dev)
        return failf(H2V_EINVAL, "%s: the program is resident on device %d, the key on device %d", who, p->dev, dev);
    if (!p->uploaded) {
        p->dev = dev;
        H2V_TRY(upload(p, st));
    }
    p->adv.release();
    p->inst.release();
    std::fill(t_last_ms, t_last_ms + 3, 0.0);
    *held = p->in.cap + p->vals.cap + p->err.cap;
    return H2V_OK;
}
size_t witness_eval_bytes(const h2v_witness_program *p) { return sizeof(fe) * (p->plan.n_inputs * 2 + p->n_computed) + 8; }
int witness_generate_dev(h2v_witness_program *p, cudaStream_t st, size_t B, const uint64_t *inputs, fe *adv, fe *inst, size_t inst_stride,
                         uint64_t *inst_host, size_t *bad_w) {
    *bad_w = B;
    H2V_TRY(ensure_eval(p, B));
    uint64_t code = 0;
    H2V_TRY(run_group(p, st, B, inputs, adv, inst, inst_stride, nullptr, inst_host, bad_w, &code, t_last_ms));
    if (*bad_w < B) return failf(H2V_EINVAL, "%s (cell %llu)", werr_text((uint32_t)(code & 255)), (unsigned long long)(code >> 8));
    return H2V_OK;
}
int witness_program_make(WitnessPlan &&plan, h2v_witness_program **out) {
    h2v_witness_program *p = new (std::nothrow) h2v_witness_program();
    if (!p) return failf(H2V_ENOMEM, "witness_program_new: out of host memory");
    p->plan = std::move(plan);
    p->n_computed = p->plan.rules.size();
    *out = p;
    return H2V_OK;
}
}  // namespace h2v

extern "C" {

void h2v_witness_program_free(h2v_witness_program_t p) {
    if (!p) return;
    if (p->uploaded && cudaSetDevice(p->dev) == cudaSuccess)
        for (DevBuf *b : {&p->rules, &p->cell_of, &p->level_start, &p->pool, &p->map, &p->in, &p->vals, &p->adv, &p->inst, &p->err}) b->release();
    delete p;
}
int h2v_witness_program_info(h2v_witness_program_t p, uint64_t out[8]) {
    if (!p || !out) return failf(H2V_EINVAL, "witness_program_info: NULL argument");
    out[0] = p->plan.n_inputs;
    out[1] = p->plan.n_cells;
    out[2] = p->n_computed;
    out[3] = p->plan.n_levels;
    out[4] = p->plan.n_adv_cols;
    out[5] = p->plan.n_instances;
    out[6] = p->plan.k;
    out[7] = p->witness_bytes();
    return H2V_OK;
}
int h2v_witness_program_rule_counts(h2v_witness_program_t p, uint64_t *out, size_t cap, size_t *n_kinds) {
    if (!p || !n_kinds) return failf(H2V_EINVAL, "witness_program_rule_counts: NULL argument");
    *n_kinds = p->plan.kind_counts.size();
    if (out) {
        if (cap < *n_kinds) return failf(H2V_EINVAL, "witness_program_rule_counts: buffer too small");
        std::copy(p->plan.kind_counts.begin(), p->plan.kind_counts.end(), out);
    }
    return H2V_OK;
}
int h2v_witness_program_inputs(h2v_witness_program_t p, uint64_t *out) {
    if (!p || (p->plan.n_inputs && !out)) return failf(H2V_EINVAL, "witness_program_inputs: NULL argument");
    std::copy(p->plan.inputs.begin(), p->plan.inputs.end(), out);
    return H2V_OK;
}
int h2v_witness_generate(h2v_witness_program_t p, size_t n_witnesses, size_t n_inputs, const uint64_t *inputs, uint64_t *advice_out,
                         uint64_t *instances_out) {
    if (!p) return failf(H2V_EINVAL, "witness_generate: NULL program");
    if (!n_witnesses) return H2V_OK;
    if (n_inputs != p->plan.n_inputs)
        return failf(H2V_EINVAL, "witness_generate: %zu inputs per witness, the program has %llu", n_inputs, (unsigned long long)p->plan.n_inputs);
    if ((n_inputs && !inputs) || !advice_out || (p->plan.n_instances && !instances_out)) return failf(H2V_EINVAL, "witness_generate: NULL argument");
    for (size_t w = 0; w < n_witnesses; ++w)
        for (size_t i = 0; i < n_inputs; ++i)
            if (!fr_reduced(inputs + 4 * (w * n_inputs + i)))
                return failf(H2V_EINVAL, "witness_generate: witness %zu: input %zu is not a reduced Montgomery value", w, i);
    std::lock_guard<std::mutex> lock(p->mu);
    const int dev = p->uploaded ? p->dev : current_device();
    if (cudaSetDevice(dev) != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ECUDA, "witness_generate: no CUDA device (libh2v has no CPU fallback)");
    }
    p->dev = dev;
    return generate(p, n_witnesses, inputs, advice_out, instances_out);
}
int h2v_witness_last_ms(double out[3]) {
    if (!out) return failf(H2V_EINVAL, "witness_last_ms: NULL argument");
    std::copy(t_last_ms, t_last_ms + 3, out);
    return H2V_OK;
}

}  // extern "C"
