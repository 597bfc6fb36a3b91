// h2v.cu -- C ABI (include/h2v.h) over the sm_100a NTT / MSM kernels: handles, workspaces,
// streams, host<->device staging.  No CPU fallback: every compute entry point needs a CUDA device.
//
// Host-side mirror of the upstream objects this library stands in for (SURVEY.md 8(a)/(b)):
//   h2v_srs     <-> halo2-axiom poly/kzg/commitment.rs ParamsKZG            (scaffold mod.rs:260)
//   h2v_domain  <-> halo2-axiom poly/domain.rs EvaluationDomain             (scaffold mod.rs:273,296)
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "h2v.h"
#include "internal.hpp"
#include "msm.cuh"
#include "ntt.cuh"
#include "poly.cuh"
#include "quotient.cuh"
#include "lookup.cuh"
#include "poseidon.hpp"

using namespace h2v;

namespace {

thread_local std::string g_err;
// The devices this process drives (h2v_init): handles hold one replica per device, `_dev` entry points run on the device
// that owns their buffers, host-facing batch entry points split their columns across all of them.  Every entry point
// picks its device once and passes it down; g_devs[0] is the primary device.
#define H2V_MAX_DEV 16
std::vector<int> g_devs = {0};
// the device a device pointer lives on (the primary one for anything the runtime does not know)
int device_of(const void *p) {
    cudaPointerAttributes at;
    if (!p || cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return g_devs[0];
    }
    return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) ? at.device : g_devs[0];
}
std::atomic<uint64_t> g_launches{0};
// device-side timing of the calling thread's last `_dev` call (per thread: concurrent callers do not mix their records)
thread_local float g_last_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
// sorted bucket entries (= mixed additions msm_accumulate executes) of the calling thread's last timed commit
thread_local uint32_t t_entry_counts[64];
thread_local int t_entry_launches = 0;
thread_local uint64_t g_last_entries = 0;
}  // namespace
// shared with the other translation units of the library (internal.hpp)
namespace h2v {
int set_error(int code, const char *msg) {
    g_err = msg;
    return code;
}
void count_launches(uint64_t n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int current_device() { return g_devs[0]; }
}  // namespace h2v
namespace {
struct MsmWorkspace {
    DevBuf buf;
};
// The polynomial primitives' stream and buffers on one device (their calls serialise on mu)
struct PolyCtx {
    std::mutex mu;
    cudaStream_t st = nullptr;
    DevBuf a, b, c, d, e, tree;
};
// What the calls without a handle keep on one device: the polynomial primitives, the MSM over caller-supplied bases
// (h2v_best_multiexp, h2v_g1_sum), h2v_best_fft, and the kernel attributes set once per device
struct DevCtx {
    PolyCtx poly;
    struct {
        std::mutex mu;
        MsmWorkspace ws;
        DevBuf sc, pts, outb;
        cudaStream_t st = nullptr;
    } raw;
    struct {
        std::mutex mu;
        DevBuf A, B, TW;
        cudaStream_t st = nullptr;
        fe cached_omega;
        int cached_L = -1;
    } fft;
    std::once_flag ntt_attr, tree_attr;
};
// One DevCtx per visible device: a `_dev` call runs on the device that owns its buffers, listed in h2v_init or not.
// NULL (error recorded) for an ordinal outside the table.
DevCtx *dev_ctx(int dev) {
    static std::vector<DevCtx> table(std::max(0, h2v_device_count()));
    if (dev >= 0 && dev < (int)table.size()) return &table[dev];
    failf(H2V_EINVAL, "device %d is not a visible CUDA device", dev);
    return nullptr;
}
// make `dev` the calling thread's device; *cx <- its DevCtx when asked for
int use_device(int dev, DevCtx **cx = nullptr) {
    cudaError_t e = cudaSetDevice(dev);
    if (e != cudaSuccess) return failf(H2V_ECUDA, "cudaSetDevice(%d): %s (libh2v has no CPU fallback)", dev, cudaGetErrorString(e));
    if (cx && !(*cx = dev_ctx(dev))) return H2V_EINVAL;
    return H2V_OK;
}

// Column staging between caller-owned host columns and a device staging area: columns that are adjacent in host memory
// (one Vec / tensor holding a whole batch) and land contiguously on the device move as ONE copy -- fewer, larger DMA
// transfers keep a PCIe link busier, most visibly when several GPUs pull from the same host at once.
// to_device: dev[c * dev_stride ..] <- host[c];  else host[c] <- dev[c * dev_stride ..];  `len` elements per column
cudaError_t stage_columns(bool to_device, fe *dev, size_t dev_stride, const uint64_t *const *host, size_t cols, size_t len, cudaStream_t st) {
    if (!len) return cudaSuccess;
    size_t c = 0;
    while (c < cols) {
        size_t run = 1;
        if (dev_stride == len)
            while (c + run < cols && host[c + run] == host[c + run - 1] + 4 * len) ++run;
        cudaError_t e = to_device ? cudaMemcpyAsync(dev + c * dev_stride, host[c], run * len * sizeof(fe), cudaMemcpyHostToDevice, st)
                                  : cudaMemcpyAsync(const_cast<uint64_t *>(host[c]), dev + c * dev_stride, run * len * sizeof(fe), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return e;
        c += run;
    }
    return cudaSuccess;
}

struct Timer {   // CUDA-event stopwatch on one stream, accumulating per kernel class
    cudaStream_t st;
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> spans;
    explicit Timer(cudaStream_t s) : st(s) {}
    Timer(const Timer &) = delete;
    Timer &operator=(const Timer &) = delete;
    ~Timer() {   // error paths return before collect(): do not leak the events
        for (auto &s : spans) {
            cudaEventDestroy(s.second.first);
            cudaEventDestroy(s.second.second);
        }
    }
    void begin(int cls) {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, st);
        spans.push_back({cls, {a, b}});
    }
    void end() { cudaEventRecord(spans.back().second.second, st); }
    void collect(bool reset) {   // call after the stream is synchronised
        if (reset)
            for (float &v : g_last_ms) v = 0;
        for (auto &s : spans) {
            float ms = 0;
            cudaEventElapsedTime(&ms, s.second.first, s.second.second);
            g_last_ms[s.first] += ms;
            cudaEventDestroy(s.second.first);
            cudaEventDestroy(s.second.second);
        }
        spans.clear();
    }
};

// A synchronous `_dev` call: enqueue(tm) on `st` (created on first use) under `mu`, then wait for the stream.  The
// device time of the call is recorded for h2v_last_kernel_ms as kernel class `cls`, or, with cls < 0, in the spans
// enqueue records on `tm` itself.  An error of enqueue wins over a CUDA error of the stream.
template <class Fn> int sync_call(std::mutex &mu, cudaStream_t &st, int cls, const char *what, Fn enqueue) {
    std::lock_guard<std::mutex> lk(mu);
    if (!st) H2V_CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    Timer tm(st);
    if (cls >= 0) tm.begin(cls);
    int rc = enqueue(tm);
    if (cls >= 0) tm.end();
    cudaError_t e = cudaStreamSynchronize(st);
    tm.collect(true);
    if (rc) return rc;
    if (e != cudaSuccess) return failf(H2V_ECUDA, "%s: %s", what, cudaGetErrorString(e));
    return H2V_OK;
}

// The lane of a small host-facing call on replica `r`, locked: the lowest free one (a single-threaded caller keeps reusing
// lane 0 and its buffers), else the next one in round-robin order.
template <class Rep> typename Rep::Lane *lock_lane(Rep *r) {
    for (auto &ln : r->lanes)
        if (ln.mu.try_lock()) return &ln;
    typename Rep::Lane *ln = &r->lanes[r->next_lane.fetch_add(1) % Rep::H2V_LANES];
    ln->mu.lock();
    return ln;
}

// ================================================================== NTT host side
const size_t NTT_SMEM_BYTES = (2 * 2048 + H2V_NTT_PLANE_PAD) * 16;

struct NttPlan {
    int P;
    int S[4];
};
NttPlan ntt_plan(int L) {
    NttPlan pl;
    pl.P = (L + 8) / 9;
    if (pl.P < 1) pl.P = 1;
    int base = L / pl.P, rem = L % pl.P;
    for (int i = 0; i < pl.P; ++i) pl.S[i] = base + (i < rem ? 1 : 0);
    return pl;
}

// dst != src, both on device `dev`.  Columns are independent; pass 0 goes src -> dst, later passes run in place on dst.
int run_ntt(int dev, cudaStream_t st, const fe *src, size_t src_stride, fe *dst, size_t dst_stride, int L, const fe *tw,
            const fe *pre, uint32_t pre_mod, uint32_t n_in, const fe *post, uint32_t post_mod, uint32_t n_out,
            size_t n_cols, uint32_t post_shift = 0) {
    if (n_cols == 0) return H2V_OK;
    if ((const void *)src == (const void *)dst) return failf(H2V_EINVAL, "run_ntt: in-place transform needs distinct buffers");
    DevCtx *cx = dev_ctx(dev);
    if (!cx) return H2V_EINVAL;
    std::call_once(cx->ntt_attr, [] {      // function attributes are per device
        cudaFuncSetAttribute(ntt_pass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NTT_SMEM_BYTES);
        cudaFuncSetAttribute(ntt_pass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)NTT_SMEM_BYTES);
    });
    NttPass p;
    memset(&p, 0, sizeof p);
    p.tw = tw;
    p.tws = tw + (L >= 1 ? ((size_t)1 << (L - 1)) : 1);      // build_twiddles: the Shoup pairs follow the Montgomery table
    p.pre = pre;
    p.pre_mod = pre_mod ? pre_mod : 1;
    p.post = post;
    p.post_mod = post_mod ? post_mod : 1;
    p.post_shift = (L > 2 && post_shift >= 3 && post_shift <= 31) ? post_shift : 0;      // else the table entry `post`
    if (p.post_shift) p.post = nullptr;
    p.n_in = n_in;
    p.n_out = n_out;
    p.L = L;
    p.src_stride = src_stride;
    p.dst_stride = dst_stride;
    for (size_t c0 = 0; c0 < n_cols; c0 += 32768) {
        unsigned cols = (unsigned)std::min<size_t>(32768, n_cols - c0);
        p.src = src + c0 * src_stride;
        p.dst = dst + c0 * dst_stride;
        if (L <= 2) {
            p.first = p.last = 1;
            ntt_tiny_kernel<<<cols, 32, 0, st>>>(p);
            H2V_LAUNCHED();
            continue;
        }
        NttPlan pl = ntt_plan(L);
        int t0 = 0;
        for (int i = 0; i < pl.P; ++i) {
            int S = pl.S[i];
            p.S = S;
            p.t0 = t0;
            p.first = (i == 0);
            p.last = (i == pl.P - 1);
            static const int loge = [] {   // log2 of the elements per CTA tile (H2V_NTT_LOGE: tuning)
                const char *e = getenv("H2V_NTT_LOGE");
                int v = e ? atoi(e) : 10;
                return v < 9 ? 9 : v > 11 ? 11 : v;
            }();
            p.logT = p.first ? std::min(loge - S, L - S) : std::min(loge - S, t0);
            if (p.logT < 0) p.logT = 0;
            unsigned threads = 1u << (S + p.logT - 3);
            unsigned tiles = 1u << (L - S - p.logT);
            size_t smem = ((size_t)2 * (1u << (S + p.logT)) + H2V_NTT_PLANE_PAD) * 16;
            static const int shoup_max_l = [] {      // H2V_NTT_SHOUP_MAX_L: tuning (0 = never, 30 = always)
                const char *e = getenv("H2V_NTT_SHOUP_MAX_L");
                return e ? atoi(e) : 18;
            }();
            if (L <= shoup_max_l) ntt_pass_kernel<true><<<dim3(tiles, cols), threads, smem, st>>>(p);
            else ntt_pass_kernel<false><<<dim3(tiles, cols), threads, smem, st>>>(p);
            H2V_LAUNCHED();
            t0 += S;
        }
    }
    return H2V_OK;
}

int build_twiddles(cudaStream_t st, DevBuf &buf, const fe &omega, int L) {
    size_t half = L >= 1 ? ((size_t)1 << (L - 1)) : 1;
    int rc = buf.ensure(3 * std::max<size_t>(half, 1) * sizeof(fe));      // Montgomery table, then (w, w') pairs
    if (rc) return rc;
    TwiddleParams tp;
    memset(&tp, 0, sizeof tp);
    fe w = omega;
    for (int b = 0; b < 28; ++b) {
        tp.pows[b] = w;
        w = fe_sqr<Fr>(w);
    }
    tp.half_n = (uint32_t)half;
    twiddle_kernel<<<(unsigned)((half + 255) / 256), 256, 0, st>>>(buf.as<fe>(), tp);
    H2V_LAUNCHED();
    return H2V_OK;
}

fe fe_from_u64x4(const uint64_t *l) {
    fe r;
    memcpy(r.v, l, 32);
    return r;
}
void fe_to_u64x4(const fe &a, uint64_t *l) { memcpy(l, a.v, 32); }
fe fr_from_small(uint64_t x) {
    fe c = fe_zero();
    c.v[0] = (uint32_t)x;
    c.v[1] = (uint32_t)(x >> 32);
    return fe_to_mont<Fr>(c);
}

// Fr::ROOT_OF_UNITY (order 2^28) and Fr::ZETA, canonical -- SURVEY.md App. B
const uint32_t FR_ROOT[8] = {0x60c37c9cu, 0xd34f1ed9u, 0xd39329c8u, 0x3215cf6du, 0x3dd31f74u, 0x98865ea9u, 0x166d18b7u, 0x03ddb9f5u};
const uint32_t FR_ZETA[8] = {0x36636f23u, 0xb8ca0b2du, 0xec2bc5e9u, 0xcc37a73fu, 0x3fd84104u, 0x048b6e19u, 0xe131a029u, 0x30644e72u};
const int FR_S = 28;

}  // namespace

struct DomRep {
    int dev = 0;
    uint32_t j, k, ek, nt;
    fe omega, omega_inv, ext_omega, ext_omega_inv, g_coset, g_coset_inv, ifft_divisor, ext_ifft_divisor;
    fe t_eval[64];
    // device constants: [0..2] coset-in (1, z, z^2); [3] ifft_divisor; [4..6] ext_ifft_divisor * (1, z^2, z);
    // [8 .. 8+nt) t_evaluations
    DevBuf dconst;
    DevBuf tw[4];   // 0: omega, 1: omega_inv, 2: ext_omega, 3: ext_omega_inv
    bool tw_ready[4] = {false, false, false, false};
    DevBuf stage_a, stage_b, pipe_a, pipe_b, pipe_a2, pipe_b2;
    DevBuf peer_in, peer_out;      // columns of another device's batch (h2v_domain_transform_dev with several devices)
    DevBuf qargs;                  // a quotient entry point's per-proof scalars and column table (under mu)
    cudaStream_t stream = nullptr, pipe_stream = nullptr, pipe_stream2 = nullptr;
    std::mutex mu, tw_mu, peer_mu;
    struct Lane {            // small host-facing transforms from concurrent caller threads (see SrsRep::Lane)
        std::mutex mu;
        cudaStream_t st = nullptr;
        DevBuf stage_a, stage_b;
    };
    static const int H2V_LANES = 4;
    Lane lanes[H2V_LANES];
    std::atomic<unsigned> next_lane{0};
};
// public handle: one replica per device
struct h2v_domain {
    std::vector<DomRep *> rep;
};

namespace {
DomRep *dom_on(h2v_domain *h, int dev) {
    for (DomRep *r : h->rep)
        if (r->dev == dev) return r;
    return nullptr;
}
// the replica a call on `h` runs on: the one on the device that holds `ptr`, the primary one for host columns
// (ptr = NULL).  NULL (error recorded) when there is none.
DomRep *dom_rep(h2v_domain *h, const void *ptr) {
    if (!h) {
        failf(H2V_EINVAL, "NULL domain");
        return nullptr;
    }
    DomRep *r = ptr ? dom_on(h, device_of(ptr)) : h->rep[0];
    if (!r) failf(H2V_EINVAL, "the columns live on device %d, which is not in the h2v_init list", device_of(ptr));
    return r;
}

// twiddle tables are built once per domain and direction, synchronously, so that any stream may use them
int domain_twiddles(DomRep *d, int which, const fe **out) {
    std::lock_guard<std::mutex> lk(d->tw_mu);
    if (!d->tw_ready[which]) {
        const fe &w = which == 0 ? d->omega : which == 1 ? d->omega_inv : which == 2 ? d->ext_omega : d->ext_omega_inv;
        int rc = build_twiddles(d->stream, d->tw[which], w, which < 2 ? (int)d->k : (int)d->ek);
        if (rc) return rc;
        H2V_CU(cudaStreamSynchronize(d->stream));
        d->tw_ready[which] = true;
    }
    *out = d->tw[which].as<fe>();
    return H2V_OK;
}

// enqueue one EvaluationDomain transform on device-resident columns
int domain_op_dev(DomRep *d, cudaStream_t st, int op, const fe *in, size_t in_stride, fe *out, size_t out_stride, size_t n_cols) {
    const fe *tw;
    const fe *dc = d->dconst.as<fe>();
    const uint32_t n = 1u << d->k, en = 1u << d->ek;
    int rc;
    switch (op) {
    case H2V_OP_LAGRANGE_TO_COEFF:
        if ((rc = domain_twiddles(d, 1, &tw))) return rc;
        return run_ntt(d->dev, st, in, in_stride, out, out_stride, d->k, tw, nullptr, 1, n, dc + 3, 1, n, n_cols, (uint32_t)d->k);      // 1/n = 2^-k
    case H2V_OP_COEFF_TO_LAGRANGE:
        if ((rc = domain_twiddles(d, 0, &tw))) return rc;
        return run_ntt(d->dev, st, in, in_stride, out, out_stride, d->k, tw, nullptr, 1, n, nullptr, 1, n, n_cols);
    case H2V_OP_COEFF_TO_EXTENDED:
        if ((rc = domain_twiddles(d, 2, &tw))) return rc;
        return run_ntt(d->dev, st, in, in_stride, out, out_stride, d->ek, tw, dc, 3, n, nullptr, 1, en, n_cols);
    case H2V_OP_EXTENDED_TO_COEFF:
        if ((rc = domain_twiddles(d, 3, &tw))) return rc;
        return run_ntt(d->dev, st, in, in_stride, out, out_stride, d->ek, tw, nullptr, 1, en, dc + 4, 3, n * (d->j - 1), n_cols);
    case H2V_OP_DIVIDE_BY_VANISHING:
        if ((rc = domain_twiddles(d, 3, &tw))) return rc;
        return run_ntt(d->dev, st, in, in_stride, out, out_stride, d->ek, tw, dc + 8, d->nt, en, dc + 4, 3, n * (d->j - 1), n_cols);
    default:
        return failf(H2V_EINVAL, "unknown domain op %d", op);
    }
}
size_t op_in_len(const DomRep *d, int op) {
    return (op == H2V_OP_EXTENDED_TO_COEFF || op == H2V_OP_DIVIDE_BY_VANISHING) ? ((size_t)1 << d->ek) : ((size_t)1 << d->k);
}
size_t op_out_len(const DomRep *d, int op) {
    if (op == H2V_OP_COEFF_TO_EXTENDED) return (size_t)1 << d->ek;
    if (op == H2V_OP_EXTENDED_TO_COEFF || op == H2V_OP_DIVIDE_BY_VANISHING) return ((size_t)1 << d->k) * (d->j - 1);
    return (size_t)1 << d->k;
}

// ================================================================== MSM host side
struct MsmCfg {
    uint32_t c, W, G;
};
uint32_t windows_for(uint32_t c) { return (255 + c - 1) / c; }
// cost model in group additions per column (SURVEY.md 8(d)): bucket adds + ~3 per bucket for the reduction
MsmCfg choose_cfg(size_t n, bool precomp) {
    MsmCfg best = {3, 85, precomp ? 1u : 85u};
    double best_cost = 1e300;
    for (uint32_t c = 3; c <= 22; ++c) {
        uint32_t W = windows_for(c);
        double nb = (double)(1u << (c - 1));
        // cost of one bucket in the reduction, in bucket additions.  Measured: 3 fits large n; at 2^16 the value 5
        // (c = 15 instead of 16) costs uniform columns 1 % and saves witness-shaped columns 10 % and single-column
        // latency 5 %; at 2^20 it loses (c = 19: 14.2 vs 12.9 ms per 4 columns).  H2V_RED_WEIGHT: tuning.
        static const double forced_w = [] {
            const char *e = getenv("H2V_RED_WEIGHT");
            return e ? atof(e) : 0.0;
        }();
        const double wred = forced_w > 0 ? forced_w : (n < ((size_t)1 << 18) ? 5.0 : 3.0);
        double cost = precomp ? (double)W * n + wred * nb : (double)W * (n + wred * nb) + 10.0 * c * W;
        if (cost < best_cost) {
            best_cost = cost;
            best = {c, W, precomp ? 1u : W};
        }
    }
    return best;
}
void fill_kadd(MsmShape &sh) {
    // K = sum_{j<W} (2^(c-1) - 1) << (j c), as 9 x 32-bit limbs
    uint32_t k[10] = {0};
    uint64_t half = ((uint64_t)1 << (sh.c - 1)) - 1;
    for (uint32_t j = 0; j < sh.W; ++j) {
        uint32_t bit = j * sh.c, w = bit >> 5, s = bit & 31;
        // add half << s at limb w (half < 2^21, so it spans at most 2 limbs)
        unsigned __int128 v = (unsigned __int128)half << s;
        uint64_t carry = 0;
        for (uint32_t q = w; q < 10; ++q) {
            uint64_t add = (uint64_t)(uint32_t)(v & 0xffffffffu);
            v >>= 32;
            uint64_t sum = (uint64_t)k[q] + add + carry;
            k[q] = (uint32_t)sum;
            carry = sum >> 32;
            if (v == 0 && carry == 0) break;
        }
    }
    for (int i = 0; i < 9; ++i) sh.kadd[i] = k[i];
}

struct Carver {
    char *base;
    size_t off = 0;
    explicit Carver(void *b) : base((char *)b) {}
    template <class T> T *take(size_t count) {
        off = (off + 255) & ~(size_t)255;
        T *p = reinterpret_cast<T *>(base + off);
        off += count * sizeof(T);
        return p;
    }
};
// sorted entries per accumulate thread: long enough that the per-chunk edge merge (one full add) is
// amortised, short enough that a single small MSM still fills the GPU.  H2V_CHUNK overrides (tuning).
std::atomic<int> g_tune_chunk{-2}, g_tune_table{-2};   // -2: read the environment on first use; -1: automatic
int tuning(std::atomic<int> &slot, const char *env) {
    int v = slot.load();
    if (v == -2) {
        const char *e = getenv(env);
        v = e ? atoi(e) : -1;
        slot.store(v);
    }
    return v;
}
// run_msm snapshots the knob once per call (h2v_set_tuning from another thread must not change the workspace layout
// between the sizing pass and the launches)
thread_local int t_tune_chunk = -1;
uint32_t pick_chunk(uint64_t entries) {
    const int forced = t_tune_chunk;
    if (forced > 0) return (uint32_t)forced;
    // small inputs are latency-bound: chunk * t(mixed add) in the accumulate thread against
    // (bucket load / chunk) * t(full add) in the finish thread is flattest around 12..24 (measured)
    uint64_t c = entries / (148ull * 2048ull);
    if (c < 12) c = 12;
    if (c > 64) c = 64;
    return (uint32_t)c;
}
struct MsmLayout {
    size_t bytes;
    uint32_t *counts, *offsets, *cursor, *tile_sums, *long_list, *long_count, *strad_count, *density;
    uint2 *entries, *strad_list;
    xyzz *buckets, *edges, *S[2], *A[2];
    uint32_t nthreads, n_buckets, l1;
};
MsmLayout msm_layout(void *base, const MsmShape &sh, uint32_t cols) {
    MsmLayout L;
    memset(&L, 0, sizeof L);
    Carver cv(base);
    uint64_t ent = (uint64_t)cols * sh.W * sh.n;
    L.n_buckets = cols * sh.G * sh.nb;
    L.nthreads = (uint32_t)((ent + sh.chunk - 1) / sh.chunk);
    // the reduction levels use segments of 8..32 (2 or 4 for a handful of buckets): size for the worst case
    L.l1 = sh.nb <= 64 ? sh.nb : (sh.nb + 7) / 8;
    size_t l2 = L.l1 <= 64 ? L.l1 : (L.l1 + 7) / 8;
    // counters cleared by ONE memset per launch: histogram, long-bucket count, straddler count, density sample
    L.counts = cv.take<uint32_t>((size_t)L.n_buckets + 8);
    L.long_count = L.counts + L.n_buckets;
    L.strad_count = L.counts + L.n_buckets + 1;
    L.density = L.counts + L.n_buckets + 2;
    L.long_list = cv.take<uint32_t>((size_t)L.nthreads / H2V_LONG_SPAN + 2);
    L.strad_list = cv.take<uint2>((size_t)L.nthreads + 1);
    L.offsets = cv.take<uint32_t>((size_t)L.n_buckets + 1);
    L.cursor = cv.take<uint32_t>(L.n_buckets);
    L.tile_sums = cv.take<uint32_t>((size_t)L.n_buckets / H2V_SCAN_TILE + 2);
    L.entries = cv.take<uint2>(ent);
    L.buckets = cv.take<xyzz>(L.n_buckets);
    L.edges = cv.take<xyzz>((size_t)2 * L.nthreads);
    L.S[0] = cv.take<xyzz>((size_t)cols * sh.G * L.l1);
    L.A[0] = cv.take<xyzz>((size_t)cols * sh.G * L.l1);
    L.S[1] = cv.take<xyzz>((size_t)cols * sh.G * l2);
    L.A[1] = cv.take<xyzz>((size_t)cols * sh.G * l2);
    L.bytes = cv.off + 256;
    return L;
}

const size_t MSM_WS_BUDGET = (size_t)16 << 30;   // per handle; columns per launch are sized to fit

// the two passes over the scalars are instantiated per window size (compile-time limb indices and shifts)
template <int C> struct WindowDispatch {
    static bool count(uint32_t c, dim3 grid, cudaStream_t st, const fe *sc, size_t stride, uint32_t *counts, const MsmShape &sh) {
        if (c == (uint32_t)C) {
            msm_count_kernel<C><<<grid, 256, 0, st>>>(sc, stride, counts, sh);
            return true;
        }
        return WindowDispatch<C - 1>::count(c, grid, st, sc, stride, counts, sh);
    }
    static bool scatter(uint32_t c, dim3 grid, cudaStream_t st, const fe *sc, size_t stride, uint32_t *cursor, uint2 *entries, const MsmShape &sh,
                        uint32_t lo, uint32_t hi) {
        if (c == (uint32_t)C) {
            msm_scatter_kernel<C><<<grid, 256, 0, st>>>(sc, stride, cursor, entries, sh, lo, hi);
            return true;
        }
        return WindowDispatch<C - 1>::scatter(c, grid, st, sc, stride, cursor, entries, sh, lo, hi);
    }
};
template <> struct WindowDispatch<2> {
    static bool count(uint32_t, dim3, cudaStream_t, const fe *, size_t, uint32_t *, const MsmShape &) { return false; }
    static bool scatter(uint32_t, dim3, cudaStream_t, const fe *, size_t, uint32_t *, uint2 *, const MsmShape &, uint32_t, uint32_t) { return false; }
};
bool launch_count(uint32_t c, dim3 grid, cudaStream_t st, const fe *sc, size_t stride, uint32_t *counts, const MsmShape &sh) {
    return WindowDispatch<24>::count(c, grid, st, sc, stride, counts, sh);
}
bool launch_scatter(uint32_t c, dim3 grid, cudaStream_t st, const fe *sc, size_t stride, uint32_t *cursor, uint2 *entries, const MsmShape &sh,
                    uint32_t lo, uint32_t hi) {
    return WindowDispatch<24>::scatter(c, grid, st, sc, stride, cursor, entries, sh, lo, hi);
}

MsmShape make_shape(size_t len, const MsmCfg &cfg, size_t pstride) {
    MsmShape sh;
    memset(&sh, 0, sizeof sh);
    sh.n = (uint32_t)len;
    sh.c = cfg.c;
    sh.W = cfg.W;
    sh.G = cfg.G;
    sh.nb = 1u << (cfg.c - 1);
    sh.pstride = (uint32_t)pstride;
    fill_kadd(sh);
    return sh;
}

// d_scalars: n_cols columns of `len` Fr (Montgomery), col_stride apart, on device `dev`.  points: bases (raw) or
// window tables (precomputed, level stride `pstride`).  Results: affine and/or Jacobian per column.
// `density` in (0, 1]: expected share of non-zero digits (sizes the accumulate chunks; 1 = uniform scalars).
int run_msm(int dev, cudaStream_t st, MsmWorkspace &ws, const fe *d_scalars, size_t col_stride, size_t n_cols, size_t len,
            const affine *points, MsmCfg cfg, size_t pstride, affine *d_out_aff, jacobian *d_out_jac, Timer *tm, double density = 1.0) {
    if (n_cols == 0) return H2V_OK;
    if (len == 0) {   // empty sum = identity: affine (0, 0); Jacobian (0, 1, 0) as halo2curves `G1::identity()`
        if (d_out_aff) H2V_CU(cudaMemsetAsync(d_out_aff, 0, n_cols * sizeof(affine), st));
        if (d_out_jac) {
            std::vector<jacobian> id(n_cols);
            for (auto &j : id) { j.x = fe_zero(); j.y = fe_one<Fq>(); j.z = fe_zero(); }
            H2V_CU(cudaMemcpyAsync(d_out_jac, id.data(), n_cols * sizeof(jacobian), cudaMemcpyHostToDevice, st));
            H2V_CU(cudaStreamSynchronize(st));
        }
        return H2V_OK;
    }
    t_tune_chunk = tuning(g_tune_chunk, "H2V_CHUNK");
    MsmShape sh = make_shape(len, cfg, pstride);
    if (!(density > 0.0) || density > 1.0) density = 1.0;
    // columns per launch: workspace budget, 2^31 entries, grid.z
    size_t max_cols = std::min<size_t>(n_cols, 16384);
    auto chunk_for = [&](size_t cols) { return pick_chunk((uint64_t)((double)cols * sh.W * sh.n * density)); };
    while (max_cols > 1) {
        sh.chunk = chunk_for(max_cols);
        MsmLayout probe = msm_layout(nullptr, sh, (uint32_t)max_cols);
        uint64_t ent = (uint64_t)max_cols * sh.W * sh.n;
        uint64_t nbk = (uint64_t)max_cols * sh.G * sh.nb;
        if (probe.bytes <= MSM_WS_BUDGET && ent < (1ull << 31) && nbk < (1ull << 31)) break;
        max_cols = (max_cols + 1) / 2;
    }
    sh.chunk = chunk_for(max_cols);
    {
        MsmLayout probe = msm_layout(nullptr, sh, (uint32_t)max_cols);
        uint64_t ent = (uint64_t)max_cols * sh.W * sh.n;
        if (ent >= (1ull << 32) - 64) return failf(H2V_EINVAL, "MSM too large: %llu bucket entries", (unsigned long long)ent);
        int rc = ws.buf.ensure(probe.bytes);
        if (rc) return rc;
    }
    DevCtx *cx = dev_ctx(dev);
    if (!cx) return H2V_EINVAL;
    std::call_once(cx->tree_attr, [] {
        cudaFuncSetAttribute(msm_reduce_tree_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * H2V_TREE_MAX * sizeof(xyzz)));
    });
    for (size_t c0 = 0; c0 < n_cols; c0 += max_cols) {
        uint32_t cols = (uint32_t)std::min(max_cols, n_cols - c0);
        sh.n_cols = cols;
        sh.chunk = chunk_for(cols);
        MsmLayout L = msm_layout(ws.buf.p, sh, cols);
        const fe *sc = d_scalars + c0 * col_stride;
        H2V_CU(cudaMemsetAsync(L.counts, 0, ((size_t)L.n_buckets + 8) * sizeof(uint32_t), st));
        unsigned gx = (unsigned)((len + 255) / 256);
        if (tm) tm->begin(0);
        if (!launch_count(sh.c, dim3(gx, cols), st, sc, col_stride, L.counts, sh)) return failf(H2V_EINVAL, "MSM window size %u unsupported", sh.c);
        H2V_LAUNCHED();
        if (tm) { tm->end(); tm->begin(1); }
        {
            const uint32_t ntiles = (L.n_buckets + H2V_SCAN_TILE - 1) / H2V_SCAN_TILE;
            msm_scan_tiles_kernel<<<ntiles, 256, 0, st>>>(L.counts, L.tile_sums, L.n_buckets);
            H2V_LAUNCHED();
            msm_scan_top_kernel<<<1, 256, 0, st>>>(L.tile_sums, ntiles, L.offsets + L.n_buckets);
            H2V_LAUNCHED();
            msm_scan_apply_kernel<<<ntiles, 256, 0, st>>>(L.counts, L.tile_sums, L.offsets, L.cursor, L.n_buckets);
            H2V_LAUNCHED();
        }
        if (tm && t_entry_launches < 64)
            H2V_CU(cudaMemcpyAsync(&t_entry_counts[t_entry_launches++], L.offsets + L.n_buckets, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (tm) { tm->end(); tm->begin(2); }
        {
            // A single very large MSM (>= 1 GiB of sorted entries) sweeps the bucket space in 4 slices: the
            // randomly written quarter of `entries` thrashes DRAM less (2^24: 7.4 -> 5.1 ms; more slices lose
            // again to the repeated passes, smaller MSMs and batches gain nothing).  H2V_SCATTER_SLICES: tuning.
            static const uint32_t forced = [] {
                const char *e = getenv("H2V_SCATTER_SLICES");
                return e ? (uint32_t)atoi(e) : 0u;
            }();
            const uint64_t ent_bytes = (uint64_t)((double)cols * sh.W * sh.n * density) * sizeof(uint2);
            uint32_t slices = forced ? forced : ((cols == 1 && ent_bytes >= (1ull << 30)) ? 4u : 1u);
            slices = std::max(1u, std::min(slices, sh.nb));
            const uint32_t per = (sh.nb + slices - 1) / slices;
            for (uint32_t sl = 0; sl < slices; ++sl) {
                launch_scatter(sh.c, dim3(gx, cols), st, sc, col_stride, L.cursor, L.entries, sh, sl * per, std::min(sh.nb, (sl + 1) * per));
                H2V_LAUNCHED();
            }
        }
        if (tm) { tm->end(); tm->begin(3); }
        const uint32_t acc_threads = L.nthreads;
        msm_accumulate_kernel<<<(acc_threads + 127) / 128, 128, 0, st>>>(L.entries, L.offsets, L.n_buckets, points, L.buckets, L.edges, sh.chunk,
                                                                        L.strad_list, L.strad_count);
        H2V_LAUNCHED();
        if (tm) { tm->end(); tm->begin(4); }
        {
            const unsigned fg = (unsigned)std::min<uint64_t>(((uint64_t)acc_threads + 127) / 128, 148ull * 16);
            msm_finish_kernel<<<fg, 128, 0, st>>>(L.offsets, L.strad_list, L.strad_count, L.edges, L.buckets, sh.chunk, L.long_list,
                                                  L.long_count);
            H2V_LAUNCHED();
            msm_finish_long_kernel<<<148 * 2, 256, 0, st>>>(L.offsets, L.edges, L.buckets, sh.chunk, L.long_list, L.long_count);
            H2V_LAUNCHED();
        }
        if (tm) { tm->end(); tm->begin(5); }
        // reduction over each (column, group): serial radix levels while they fill the GPU, then one log-depth tree
        const uint32_t n_inst = cols * sh.G;
        const xyzz *Sin = L.buckets, *Ain = nullptr;
        const uint32_t *occ = L.offsets;
        uint32_t cnt = sh.nb, shift = 0;
        int pp = 0;
        while (cnt > 1) {
            if (cnt <= H2V_TREE_MAX && !occ) {
                const unsigned threads = std::max(32u, std::min(256u, cnt / 2));
                msm_reduce_tree_kernel<<<n_inst, threads, 2 * cnt * sizeof(xyzz), st>>>(Sin, Ain, cnt, shift, L.S[pp], L.A[pp]);
                H2V_LAUNCHED();
                Sin = L.S[pp];
                Ain = L.A[pp];
                cnt = 1;
                break;
            }
            // segments of 32 while that still fills the GPU once (each thread is a serial chain), shorter otherwise;
            // never below what brings the level to the tree's size in one step
            uint32_t log_seg = 5;
            while (log_seg > 3 && (uint64_t)n_inst * (cnt >> log_seg) < 148ull * 256 && (cnt >> (log_seg - 1)) <= H2V_TREE_MAX) --log_seg;
            while (log_seg > 1 && (cnt >> log_seg) < 2) --log_seg;
            uint32_t cnt_out = (cnt + (1u << log_seg) - 1) >> log_seg;
            uint32_t total = n_inst * cnt_out;
            msm_reduce_kernel<<<(total + 127) / 128, 128, 0, st>>>(Sin, Ain, L.S[pp], L.A[pp], cnt, cnt_out, n_inst, shift, log_seg, occ);
            H2V_LAUNCHED();
            occ = nullptr;
            Sin = L.S[pp];
            Ain = L.A[pp];
            pp ^= 1;
            cnt = cnt_out;
            shift += log_seg;
        }
        if (!Ain) {   // nb == 1: a single bucket per group, its weight is 1 and there is no weighted part
            msm_reduce_kernel<<<(n_inst + 127) / 128, 128, 0, st>>>(Sin, nullptr, L.S[pp], L.A[pp], 1, 1, n_inst, 0, 3, occ);
            H2V_LAUNCHED();
            Sin = L.S[pp];
            Ain = L.A[pp];
        }
        if (tm) { tm->end(); tm->begin(6); }
        msm_final_kernel<<<cols, 32, 0, st>>>(Sin, Ain, cols, sh.G, sh.c, d_out_aff ? d_out_aff + c0 : nullptr,
                                                          d_out_jac ? d_out_jac + c0 : nullptr);
        H2V_LAUNCHED();
        if (tm) tm->end();
    }
    return H2V_OK;
}

}  // namespace

struct SrsRep {
    int dev = 0;
    uint32_t k;
    size_t n;
    // Window tables, two per basis: [0] the window the cost model picks for uniform scalars, [1] a smaller window
    // (fewer buckets, more digits per scalar) for columns whose scalars are mostly 0 / 1 / small -- real witness
    // columns -- and for single small calls, where the bucket reduction would otherwise dominate.  W levels of n
    // affine points each (level 0 = the bases).
    DevBuf table[2][2];
    bool have[2] = {false, false};
    bool have_small = false;
    MsmCfg cfg[2];
    MsmWorkspace ws, ws2;
    DevBuf stage, out;
    DevBuf peer_in, peer_out;      // columns of another device's batch and their commitments (several devices)
    std::mutex peer_mu;               // held from the pull to the write-back
    cudaStream_t stream = nullptr, stream2 = nullptr, copy_stream = nullptr, up_stream = nullptr;
    cudaEvent_t copied[2] = {nullptr, nullptr}, computed[2] = {nullptr, nullptr};
    std::mutex mu;
    // Small calls (a single commit_lagrange from one of the caller's worker threads -- stock create_proof
    // commits column by column from a rayon pool) run on one of H2V_LANES independent lanes, each with its
    // own stream, workspace and staging, so concurrent callers overlap instead of queueing on one mutex.
    struct Lane {
        std::mutex mu;
        cudaStream_t st = nullptr;
        MsmWorkspace ws;
        DevBuf stage, out;
    };
    static const int H2V_LANES = 4;
    Lane lanes[H2V_LANES];
    std::atomic<unsigned> next_lane{0};
    int last_variant = 0;
};
struct h2v_srs {
    std::vector<SrsRep *> rep;
};

namespace {
SrsRep *srs_on(h2v_srs *h, int dev) {
    for (SrsRep *r : h->rep)
        if (r->dev == dev) return r;
    return nullptr;
}
// Window choice per call: the share of non-zero digits under both window sizes is estimated from a strided sample of
// the batch (one small kernel + a 16-byte read-back), then the cheaper plan wins under the cost model
//   10 products per bucket addition (mixed add) + 28 per bucket of the reduction (two full additions).
// Results never depend on the choice.  h2v_set_tuning(_, table) / H2V_TABLE force a table (tests).
int msm_srs(SrsRep *s, cudaStream_t st, MsmWorkspace &ws, int basis, const fe *d_scalars, size_t col_stride, size_t n_cols, size_t len,
            affine *d_out, Timer *tm) {
    int variant = 0;
    double density = 1.0;
    const int forced = tuning(g_tune_table, "H2V_TABLE");
    if (n_cols && len && s->have_small) {
        if (forced == 0 || forced == 1) {
            variant = forced;
        } else {
            const uint32_t samples = (uint32_t)std::min<uint64_t>(4096, (uint64_t)n_cols * len);
            int rc = ws.buf.ensure(4096);
            if (rc) return rc;
            uint32_t *d_cnt = ws.buf.as<uint32_t>();
            H2V_CU(cudaMemsetAsync(d_cnt, 0, 8, st));
            MsmShape s0 = make_shape(len, s->cfg[0], s->n), s1 = make_shape(len, s->cfg[1], s->n);
            msm_density_kernel<<<(samples + 255) / 256, 256, 0, st>>>(d_scalars, col_stride, (uint32_t)n_cols, (uint32_t)len, samples, s0, s1, d_cnt);
            H2V_LAUNCHED();
            uint32_t h_cnt[2] = {0, 0};
            H2V_CU(cudaMemcpyAsync(h_cnt, d_cnt, 8, cudaMemcpyDeviceToHost, st));
            H2V_CU(cudaStreamSynchronize(st));
            const double e0 = (double)h_cnt[0] / samples * len, e1 = (double)h_cnt[1] / samples * len;      // entries per column
            // the reduction is latency-bound when few columns share it: weigh it up for small batches
            const double inst_w = n_cols >= 32 ? 28.0 : 28.0 * (1.0 + 24.0 / (double)n_cols);
            const double cost0 = 10.0 * e0 + inst_w * (double)(1u << (s->cfg[0].c - 1));
            const double cost1 = 10.0 * e1 + inst_w * (double)(1u << (s->cfg[1].c - 1));
            variant = cost1 < cost0 ? 1 : 0;
            density = (variant ? e1 : e0) / ((double)s->cfg[variant].W * len);
            density = std::min(1.0, density * 1.1 + 0.01);
        }
    }
    s->last_variant = variant;
    return run_msm(s->dev, st, ws, d_scalars, col_stride, n_cols, len, s->table[basis][variant].as<affine>(), s->cfg[variant], s->n, d_out, nullptr, tm,
                   density);
}
}  // namespace

// ================================================================== C ABI
extern "C" {

const char *h2v_last_error(void) { return g_err.c_str(); }
const char *h2v_version(void) { return "h2v-b200 0.1 (sm_100a)"; }
uint64_t h2v_launch_count(void) { return g_launches.load(); }

int h2v_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
// The CUDA devices this process drives, in order; devices[0] is the primary one (handle-less and host-facing
// single-column entry points run there).  Call before creating handles.  NULL / 0 = device 0.
int h2v_init(const int *devices, int n_dev) {
    int n = h2v_device_count();
    if (n <= 0) return failf(H2V_ECUDA, "no CUDA device visible (libh2v has no CPU fallback)");
    std::vector<int> devs;
    if (!devices || n_dev <= 0) {
        devs.push_back(0);
    } else {
        if (n_dev > H2V_MAX_DEV) return failf(H2V_EINVAL, "h2v_init: at most %d devices", H2V_MAX_DEV);
        for (int i = 0; i < n_dev; ++i) {
            if (devices[i] < 0 || devices[i] >= n) return failf(H2V_EINVAL, "device %d out of range (have %d)", devices[i], n);
            for (int d : devs)
                if (d == devices[i]) return failf(H2V_EINVAL, "h2v_init: device %d listed twice", d);
            devs.push_back(devices[i]);
        }
    }
    for (int d : devs) {
        H2V_CU(cudaSetDevice(d));
        H2V_CU(cudaFree(0));
    }
    // peer access between all pairs (SRS replicas are copied device to device); failure just means staged copies
    for (int a : devs)
        for (int b : devs) {
            if (a == b) continue;
            int ok = 0;
            if (cudaDeviceCanAccessPeer(&ok, a, b) == cudaSuccess && ok) {
                cudaSetDevice(a);
                cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
                if (e != cudaSuccess) cudaGetLastError();
            }
        }
    g_devs = devs;
    H2V_CU(cudaSetDevice(g_devs[0]));
    return H2V_OK;
}
int h2v_device_list(int *out, int cap) {
    for (int i = 0; i < (int)g_devs.size() && i < cap; ++i) out[i] = g_devs[i];
    return (int)g_devs.size();
}
// Proof wire format of a commitment (SURVEY.md 8(f) row 3): halo2curves 0.3.x `G1Affine::to_bytes()` =
// canonical x, little-endian, with the parity of canonical y in the top bit of byte 31 (poseidon.hpp); identity = 32 zero bytes.
// Host-side (a proof holds ~10^3 commitments); uses the host instantiation of the field code.
int h2v_g1_to_bytes(const uint64_t *affine_pts, size_t n, uint8_t *out) {
    if (n && (!affine_pts || !out)) return failf(H2V_EINVAL, "g1_to_bytes: NULL buffer");
    for (size_t i = 0; i < n; ++i) {
        affine p;
        memcpy(&p, affine_pts + 8 * i, sizeof p);
        uint8_t *o = out + 32 * i;
        if (affine_is_identity(p)) {
            memset(o, 0, 32);
            continue;
        }
        g1_affine_to_bytes(p, o);
    }
    return H2V_OK;
}
// `Fr::to_repr()`: canonical little-endian bytes of Montgomery-form scalars
int h2v_fr_to_repr(const uint64_t *fr_mont, size_t n, uint8_t *out) {
    if (n && (!fr_mont || !out)) return failf(H2V_EINVAL, "fr_to_repr: NULL buffer");
    for (size_t i = 0; i < n; ++i) {
        fe a;
        memcpy(a.v, fr_mont + 4 * i, 32);
        fe c = fe_from_mont<Fr>(a);
        memcpy(out + 32 * i, c.v, 32);
    }
    return H2V_OK;
}
int h2v_dev_alloc(size_t bytes, void **d_out) {
    H2V_TRY(use_device(g_devs[0]));
    if (!d_out || !bytes) return failf(H2V_EINVAL, "dev_alloc: bad argument");
    cudaError_t e = cudaMalloc(d_out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ENOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
    }
    return H2V_OK;
}
int h2v_dev_free(void *d_ptr) {
    H2V_TRY(use_device(device_of(d_ptr)));
    if (d_ptr) H2V_CU(cudaFree(d_ptr));
    return H2V_OK;
}
int h2v_dev_upload(void *d_dst, const void *src, size_t bytes) {
    H2V_TRY(use_device(device_of(d_dst)));
    if (bytes && (!d_dst || !src)) return failf(H2V_EINVAL, "dev_upload: NULL buffer");
    H2V_CU(cudaMemcpy(d_dst, src, bytes, cudaMemcpyHostToDevice));
    return H2V_OK;
}
int h2v_dev_download(void *dst, const void *d_src, size_t bytes) {
    H2V_TRY(use_device(device_of(d_src)));
    if (bytes && (!dst || !d_src)) return failf(H2V_EINVAL, "dev_download: NULL buffer");
    H2V_CU(cudaMemcpy(dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return H2V_OK;
}
int h2v_host_register(void *ptr, size_t bytes) {
    H2V_TRY(use_device(g_devs[0]));
    if (!ptr || !bytes) return failf(H2V_EINVAL, "host_register: bad argument");
    H2V_CU(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    return H2V_OK;
}
int h2v_host_unregister(void *ptr) {
    H2V_TRY(use_device(g_devs[0]));
    H2V_CU(cudaHostUnregister(ptr));
    return H2V_OK;
}
int h2v_set_tuning(int chunk, int table) {
    g_tune_chunk.store(chunk > 0 ? chunk : -1);
    g_tune_table.store(table == 0 || table == 1 ? table : -1);
    return H2V_OK;
}
uint64_t h2v_last_msm_entries(void) { return g_last_entries; }
int h2v_last_kernel_ms(float out[8]) {
    if (!out) return failf(H2V_EINVAL, "last_kernel_ms: NULL");
    memcpy(out, g_last_ms, sizeof g_last_ms);
    return H2V_OK;
}

// ---------------------------------------------------------------- SRS / commit
static void rep_srs_free(SrsRep *s);
// the replica on device `dev` built from the host bases: the window tables are computed there
static int rep_srs_load(int dev, uint32_t k, const uint64_t *g, const uint64_t *g_lagrange, SrsRep **out) {
    if (k > 26) return failf(H2V_EINVAL, "h2v_srs_load: k = %u unsupported", k);
    int rc = use_device(dev);
    if (rc) return rc;
    SrsRep *s = new SrsRep();
    s->dev = dev;
    s->k = k;
    s->n = (size_t)1 << k;
    s->cfg[0] = choose_cfg(s->n, true);
    // cap the table footprint at 24 GB per basis by shrinking the number of levels (bigger windows)
    while ((size_t)s->cfg[0].W * s->n * sizeof(affine) > ((size_t)24 << 30) && s->cfg[0].c < 24) {
        s->cfg[0].c++;
        s->cfg[0].W = windows_for(s->cfg[0].c);
    }
    // second table with a window two bits smaller: a quarter of the buckets (H2V_SMALL_WINDOW_DELTA: tuning; 0 = none)
    static const int small_delta = [] {
        const char *e = getenv("H2V_SMALL_WINDOW_DELTA");
        return e ? atoi(e) : 2;
    }();
    s->cfg[1] = s->cfg[0];
    if (small_delta > 0 && (int)s->cfg[0].c - small_delta >= 3) {
        s->cfg[1].c = s->cfg[0].c - (uint32_t)small_delta;
        s->cfg[1].W = windows_for(s->cfg[1].c);
        s->have_small = (size_t)s->cfg[1].W * s->n * sizeof(affine) <= ((size_t)8 << 30);
    }
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete s;
        return failf(H2V_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    const uint64_t *src[2] = {g, g_lagrange};
    for (int b = 0; b < 2; ++b) {
        if (!src[b]) continue;
        for (int v = 0; v < (s->have_small ? 2 : 1); ++v) {
            DevBuf &tb = s->table[b][v];
            rc = tb.ensure((size_t)s->cfg[v].W * s->n * sizeof(affine));
            if (rc) { rep_srs_free(s); return rc; }
            if (v == 0) e = cudaMemcpyAsync(tb.p, src[b], s->n * sizeof(affine), cudaMemcpyHostToDevice, s->stream);
            else e = cudaMemcpyAsync(tb.p, s->table[b][0].p, s->n * sizeof(affine), cudaMemcpyDeviceToDevice, s->stream);
            if (e != cudaSuccess) { rep_srs_free(s); return failf(H2V_ECUDA, "SRS upload: %s", cudaGetErrorString(e)); }
            for (uint32_t lvl = 1; lvl < s->cfg[v].W; ++lvl) {
                msm_precompute_kernel<<<(unsigned)((s->n + 127) / 128), 128, 0, s->stream>>>(tb.as<affine>(), (uint32_t)s->n, lvl, s->cfg[v].c);
                g_launches.fetch_add(1);
            }
        }
        s->have[b] = true;
    }
    e = cudaStreamSynchronize(s->stream);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { rep_srs_free(s); return failf(H2V_ECUDA, "SRS table build: %s", cudaGetErrorString(e)); }
    *out = s;
    return H2V_OK;
}
int h2v_srs_info(h2v_srs_t h, uint32_t *window_bits, uint32_t *windows) {
    if (!h) return failf(H2V_EINVAL, "srs_info: NULL srs");
    const SrsRep *s = h->rep[0];
    // the table the last commit on this handle used (the main one before any commit)
    if (window_bits) *window_bits = s->cfg[s->last_variant].c;
    if (windows) *windows = s->cfg[s->last_variant].W;
    return H2V_OK;
}
static void rep_srs_free(SrsRep *s) {
    if (!s) return;
    cudaSetDevice(s->dev);
    for (auto &tb : s->table)
        for (auto &t : tb) t.release();
    s->ws.buf.release();
    s->ws2.buf.release();
    for (auto &ln : s->lanes) {
        ln.ws.buf.release();
        ln.stage.release();
        ln.out.release();
        if (ln.st) cudaStreamDestroy(ln.st);
    }
    s->stage.release();
    s->out.release();
    s->peer_in.release();
    s->peer_out.release();
    if (s->stream) cudaStreamDestroy(s->stream);
    if (s->up_stream) cudaStreamDestroy(s->up_stream);
    if (s->copy_stream) {
        cudaStreamDestroy(s->copy_stream);
        cudaStreamDestroy(s->stream2);
        for (int b = 0; b < 2; ++b) {
            cudaEventDestroy(s->copied[b]);
            cudaEventDestroy(s->computed[b]);
        }
    }
    delete s;
}

static int rep_commit_batch_dev(SrsRep *s, int basis, const void *d_polys, size_t col_stride, size_t n_polys, size_t len,
                         void *d_out_affine) {
    if (!s) return failf(H2V_EINVAL, "commit: NULL srs");
    if (basis != 0 && basis != 1) return failf(H2V_EINVAL, "commit: basis must be 0 or 1");
    if (!s->have[basis]) return failf(H2V_EINVAL, "commit: basis %d was not loaded", basis);
    if (len > s->n) return failf(H2V_EINVAL, "commit: poly length %zu exceeds n = %zu", len, s->n);
    if (n_polys && (!d_polys || !d_out_affine)) return failf(H2V_EINVAL, "commit: NULL buffer");
    H2V_TRY(use_device(s->dev));
    t_entry_launches = 0;
    int rc = sync_call(s->mu, s->stream, -1, "commit", [&](Timer &tm) {
        return msm_srs(s, s->stream, s->ws, basis, (const fe *)d_polys, col_stride, n_polys, len, (affine *)d_out_affine, &tm);
    });
    g_last_entries = 0;
    for (int i = 0; i < t_entry_launches; ++i) g_last_entries += t_entry_counts[i];
    return rc;
}

static int rep_commit_batch(SrsRep *s, int basis, const uint64_t *const *polys, size_t n_polys, size_t len, uint64_t *out_affine) {
    if (!s) return failf(H2V_EINVAL, "commit: NULL srs");
    if (basis != 0 && basis != 1) return failf(H2V_EINVAL, "commit: basis must be 0 or 1");
    if (!s->have[basis]) return failf(H2V_EINVAL, "commit: basis %d was not loaded", basis);
    if (len > s->n) return failf(H2V_EINVAL, "commit: poly length %zu exceeds n = %zu", len, s->n);
    if (n_polys == 0) return H2V_OK;
    if (!polys || !out_affine) return failf(H2V_EINVAL, "commit: NULL buffer");
    int rc = use_device(s->dev);
    if (rc) return rc;
    const size_t stride_small = std::max<size_t>(len, 1);
    if (n_polys * stride_small * sizeof(fe) <= ((size_t)48 << 20)) {
        // one sub-batch, on a lane
        SrsRep::Lane *ln = lock_lane(s);
        std::lock_guard<std::mutex> lk(ln->mu, std::adopt_lock);
        if (!ln->st) H2V_CU(cudaStreamCreateWithFlags(&ln->st, cudaStreamNonBlocking));
        if ((rc = ln->stage.ensure(n_polys * stride_small * sizeof(fe)))) return rc;
        if ((rc = ln->out.ensure(n_polys * sizeof(affine)))) return rc;
        for (size_t c = 0; c < n_polys; ++c)
            if (!polys[c] && len) return failf(H2V_EINVAL, "commit: polys[%zu] is NULL", c);
        H2V_CU(stage_columns(true, ln->stage.as<fe>(), stride_small, polys, n_polys, len, ln->st));
        rc = msm_srs(s, ln->st, ln->ws, basis, ln->stage.as<fe>(), stride_small, n_polys, len, ln->out.as<affine>(), nullptr);
        if (rc) {
            cudaStreamSynchronize(ln->st);
            return rc;
        }
        H2V_CU(cudaMemcpyAsync(out_affine, ln->out.p, n_polys * sizeof(affine), cudaMemcpyDeviceToHost, ln->st));
        H2V_CU(cudaStreamSynchronize(ln->st));
        return H2V_OK;
    }
    std::lock_guard<std::mutex> lk(s->mu);
    // Double-buffered staging: while the kernels of sub-batch i run, the columns of sub-batch i+1 cross PCIe
    // on `copy_stream` (effective when the caller's buffers are pinned).  Sub-batches alternate between two
    // compute streams with their own workspaces, so the latency-bound tail of one (bucket-reduction tree,
    // affine normalisation) overlaps the bulk kernels of the next.
    const size_t stride = std::max<size_t>(len, 1);
    // Sub-batch schedule: a small first sub-batch (its upload is the only one nothing can hide) and large ones
    // after it (big launches are the efficient ones; their uploads hide behind the previous launch).
    static const size_t sub_mb = [] {   // scalars per large sub-batch in MiB (H2V_SUB_MB / H2V_FIRST_MB: tuning; 400 / 32 measured best:
                                        // 96 x 2^16 end to end 21.2 -> 20.6 ms against 96 / 16 -- few, large launches amortise the reduction tails)
        const char *e = getenv("H2V_SUB_MB");
        int v = e ? atoi(e) : 400;
        return (size_t)(v < 1 ? 1 : v);
    }();
    static const size_t first_mb = [] {
        const char *e = getenv("H2V_FIRST_MB");
        int v = e ? atoi(e) : 32;
        return (size_t)(v < 1 ? 1 : v);
    }();
    size_t sub = std::max<size_t>(1, (sub_mb << 20) / (stride * sizeof(fe)));
    const size_t first = std::max<size_t>(1, std::min(sub, (first_mb << 20) / (stride * sizeof(fe))));
    sub = std::min(sub, n_polys);
    if ((rc = s->stage.ensure(2 * sub * stride * sizeof(fe)))) return rc;
    if ((rc = s->out.ensure(n_polys * sizeof(affine)))) return rc;
    if (!s->copy_stream) {
        H2V_CU(cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking));
        H2V_CU(cudaStreamCreateWithFlags(&s->stream2, cudaStreamNonBlocking));
        for (int b = 0; b < 2; ++b) {
            H2V_CU(cudaEventCreateWithFlags(&s->copied[b], cudaEventDisableTiming));
            H2V_CU(cudaEventCreateWithFlags(&s->computed[b], cudaEventDisableTiming));
        }
    }
    size_t it = 0;
    for (size_t c0 = 0, step = 0; c0 < n_polys; c0 += step, ++it) {
        step = it == 0 ? first : sub;
        const size_t cols = std::min(step, n_polys - c0);
        const int b = (int)(it & 1);
        fe *stg = s->stage.as<fe>() + (size_t)b * sub * stride;
        if (it >= 2) H2V_CU(cudaStreamWaitEvent(s->copy_stream, s->computed[b], 0));
        for (size_t c = 0; c < cols; ++c) {
            if (!polys[c0 + c] && len) {
                cudaStreamSynchronize(s->stream);
                cudaStreamSynchronize(s->copy_stream);
                return failf(H2V_EINVAL, "commit: polys[%zu] is NULL", c0 + c);
            }
        }
        H2V_CU(stage_columns(true, stg, stride, polys + c0, cols, len, s->copy_stream));
        H2V_CU(cudaEventRecord(s->copied[b], s->copy_stream));
        cudaStream_t cst = b ? s->stream2 : s->stream;
        H2V_CU(cudaStreamWaitEvent(cst, s->copied[b], 0));
        rc = msm_srs(s, cst, b ? s->ws2 : s->ws, basis, stg, stride, cols, len, s->out.as<affine>() + c0, nullptr);
        if (rc) {
            cudaStreamSynchronize(s->stream);
            cudaStreamSynchronize(s->stream2);
            cudaStreamSynchronize(s->copy_stream);
            return rc;
        }
        H2V_CU(cudaEventRecord(s->computed[b], cst));
    }
    if (it > 1) H2V_CU(cudaStreamWaitEvent(s->stream, s->computed[1], 0));
    H2V_CU(cudaMemcpyAsync(out_affine, s->out.p, n_polys * sizeof(affine), cudaMemcpyDeviceToHost, s->stream));
    H2V_CU(cudaStreamSynchronize(s->stream));
    return H2V_OK;
}

// one MSM over caller-supplied bases (no handle, no tables): Jacobian and / or affine result
static int multiexp_raw(const uint64_t *coeffs, const uint64_t *bases, size_t n, uint64_t *out_jacobian, uint64_t *out_affine) {
    const int dev = g_devs[0];
    DevCtx *cx;
    int rc = use_device(dev, &cx);
    if (rc) return rc;
    MsmWorkspace &ws = cx->raw.ws;
    DevBuf &sc = cx->raw.sc, &pts = cx->raw.pts, &outb = cx->raw.outb;
    cudaStream_t &st = cx->raw.st;
    std::lock_guard<std::mutex> lk(cx->raw.mu);
    if (!st) H2V_CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    if ((rc = sc.ensure(n * sizeof(fe)))) return rc;
    if ((rc = pts.ensure(n * sizeof(affine)))) return rc;
    if ((rc = outb.ensure(sizeof(jacobian) + sizeof(affine)))) return rc;
    H2V_CU(cudaMemcpyAsync(sc.p, coeffs, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(pts.p, bases, n * sizeof(affine), cudaMemcpyHostToDevice, st));
    MsmCfg cfg = choose_cfg(n, false);
    jacobian *dj = outb.as<jacobian>();
    affine *da = reinterpret_cast<affine *>(dj + 1);
    rc = run_msm(dev, st, ws, sc.as<fe>(), n, 1, n, pts.as<affine>(), cfg, n, out_affine ? da : nullptr, out_jacobian ? dj : nullptr, nullptr);
    if (rc) { cudaStreamSynchronize(st); return rc; }
    if (out_jacobian) H2V_CU(cudaMemcpyAsync(out_jacobian, dj, sizeof(jacobian), cudaMemcpyDeviceToHost, st));
    if (out_affine) H2V_CU(cudaMemcpyAsync(out_affine, da, sizeof(affine), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}
int h2v_best_multiexp(const uint64_t *coeffs, const uint64_t *bases, size_t n, uint64_t out_jacobian[12]) {
    if (!out_jacobian) return failf(H2V_EINVAL, "best_multiexp: NULL output");
    if (n && (!coeffs || !bases)) return failf(H2V_EINVAL, "best_multiexp: NULL input");
    if (n >= ((size_t)1 << 27)) return failf(H2V_EINVAL, "best_multiexp: n = %zu unsupported", n);
    if (n == 0) {
        H2V_TRY(use_device(g_devs[0]));
        jacobian id;      // halo2curves `G1::identity()` = (0, 1, 0)
        id.x = fe_zero(); id.y = fe_one<Fq>(); id.z = fe_zero();
        memcpy(out_jacobian, &id, 96);
        return H2V_OK;
    }
    return multiexp_raw(coeffs, bases, n, out_jacobian, nullptr);
}
int h2v_g1_sum(const uint64_t *affine_pts, size_t n, uint64_t out_affine[8]) {
    if (!out_affine) return failf(H2V_EINVAL, "g1_sum: NULL output");
    if (n && !affine_pts) return failf(H2V_EINVAL, "g1_sum: NULL input");
    if (n >= ((size_t)1 << 27)) return failf(H2V_EINVAL, "g1_sum: n = %zu unsupported", n);
    if (n == 0) {
        H2V_TRY(use_device(g_devs[0]));
        memset(out_affine, 0, 64);
        return H2V_OK;
    }
    std::vector<fe> ones(n, fe_one<Fr>());
    return multiexp_raw(reinterpret_cast<const uint64_t *>(ones.data()), affine_pts, n, nullptr, out_affine);
}

// ---------------------------------------------------------------- FFT / domain
int h2v_best_fft(uint64_t *a, const uint64_t omega[4], uint32_t log_n) {
    if (!a || !omega) return failf(H2V_EINVAL, "best_fft: NULL argument");
    if (log_n > 27) return failf(H2V_EINVAL, "best_fft: log_n = %u unsupported", log_n);
    const int dev = g_devs[0];
    DevCtx *cx;
    int rc = use_device(dev, &cx);
    if (rc) return rc;
    DevBuf &A = cx->fft.A, &B = cx->fft.B, &TW = cx->fft.TW;
    cudaStream_t &st = cx->fft.st;
    fe &cached_omega = cx->fft.cached_omega;
    int &cached_L = cx->fft.cached_L;
    std::lock_guard<std::mutex> lk(cx->fft.mu);
    if (!st) H2V_CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    size_t n = (size_t)1 << log_n;
    if ((rc = A.ensure(n * sizeof(fe)))) return rc;
    if ((rc = B.ensure(n * sizeof(fe)))) return rc;
    fe w = fe_from_u64x4(omega);
    if (cached_L != (int)log_n || !fe_eq(w, cached_omega)) {   // twiddles are kept for repeated (omega, log_n)
        if ((rc = build_twiddles(st, TW, w, (int)log_n))) return rc;
        cached_L = (int)log_n;
        cached_omega = w;
    }
    H2V_CU(cudaMemcpyAsync(A.p, a, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    rc = run_ntt(dev, st, A.as<fe>(), n, B.as<fe>(), n, (int)log_n, TW.as<fe>(), nullptr, 1, (uint32_t)n, nullptr, 1, (uint32_t)n, 1);
    if (rc) { cudaStreamSynchronize(st); return rc; }
    H2V_CU(cudaMemcpyAsync(a, B.p, n * sizeof(fe), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}

static void rep_domain_free(DomRep *d);
static int rep_domain_new(int dev, uint32_t j, uint32_t k, DomRep **out) {
    if (j < 2) return failf(H2V_EINVAL, "domain_new: j = %u (need j >= 2)", j);
    uint32_t ek = k;
    while (((uint64_t)1 << ek) < ((uint64_t)1 << k) * (j - 1)) ++ek;
    if (ek > 27 || ek - k > 6) return failf(H2V_EINVAL, "domain_new: extended_k = %u unsupported", ek);
    int rc = use_device(dev);
    if (rc) return rc;
    DomRep *d = new DomRep();
    d->dev = dev;
    d->j = j;
    d->k = k;
    d->ek = ek;
    d->nt = 1u << (ek - k);
    fe root;
    memcpy(root.v, FR_ROOT, 32);
    root = fe_to_mont<Fr>(root);
    d->ext_omega = root;
    for (uint32_t i = ek; i < (uint32_t)FR_S; ++i) d->ext_omega = fe_sqr<Fr>(d->ext_omega);
    d->omega = d->ext_omega;
    for (uint32_t i = k; i < ek; ++i) d->omega = fe_sqr<Fr>(d->omega);
    d->omega_inv = fe_inv<Fr>(d->omega);
    d->ext_omega_inv = fe_inv<Fr>(d->ext_omega);
    fe zeta;
    memcpy(zeta.v, FR_ZETA, 32);
    d->g_coset = fe_to_mont<Fr>(zeta);
    d->g_coset_inv = fe_sqr<Fr>(d->g_coset);
    d->ifft_divisor = fe_inv<Fr>(fr_from_small((uint64_t)1 << k));
    d->ext_ifft_divisor = fe_inv<Fr>(fr_from_small((uint64_t)1 << ek));
    fe cur = d->g_coset, one = fe_one<Fr>();
    for (uint32_t i = 0; i < d->nt; ++i) {
        fe v = fe_sub<Fr>(fe_pow_u64<Fr>(cur, (uint64_t)1 << k), one);
        d->t_eval[i] = fe_inv<Fr>(v);
        cur = fe_mul<Fr>(cur, d->ext_omega);
    }
    fe hc[8 + 64];
    for (auto &x : hc) x = fe_zero();
    hc[0] = one;
    hc[1] = d->g_coset;
    hc[2] = d->g_coset_inv;
    hc[3] = d->ifft_divisor;
    hc[4] = d->ext_ifft_divisor;
    hc[5] = fe_mul<Fr>(d->ext_ifft_divisor, d->g_coset_inv);
    hc[6] = fe_mul<Fr>(d->ext_ifft_divisor, d->g_coset);
    for (uint32_t i = 0; i < d->nt; ++i) hc[8 + i] = d->t_eval[i];
    cudaError_t e = cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        rc = d->dconst.ensure(sizeof hc);
        if (rc) { rep_domain_free(d); return rc; }
        e = cudaMemcpy(d->dconst.p, hc, sizeof hc, cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) {
        rep_domain_free(d);
        return failf(H2V_ECUDA, "domain_new: %s", cudaGetErrorString(e));
    }
    *out = d;
    return H2V_OK;
}
static void rep_domain_free(DomRep *d) {
    if (!d) return;
    cudaSetDevice(d->dev);
    d->dconst.release();
    for (auto &t : d->tw) t.release();
    d->stage_a.release();
    d->stage_b.release();
    d->pipe_a.release();
    d->pipe_b.release();
    d->pipe_a2.release();
    d->pipe_b2.release();
    d->peer_in.release();
    d->peer_out.release();
    if (d->pipe_stream) cudaStreamDestroy(d->pipe_stream);
    if (d->pipe_stream2) cudaStreamDestroy(d->pipe_stream2);
    for (auto &ln : d->lanes) {
        ln.stage_a.release();
        ln.stage_b.release();
        if (ln.st) cudaStreamDestroy(ln.st);
    }
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
}
uint32_t h2v_domain_k(h2v_domain_t h) { return h ? h->rep[0]->k : 0; }
uint32_t h2v_domain_extended_k(h2v_domain_t h) { return h ? h->rep[0]->ek : 0; }
int h2v_domain_constant(h2v_domain_t h, int which, uint64_t out[4]) {
    if (!h || !out) return failf(H2V_EINVAL, "domain_constant: NULL argument");
    const DomRep *d = h->rep[0];
    const fe *p = nullptr;
    switch (which) {
    case 0: p = &d->omega; break;
    case 1: p = &d->omega_inv; break;
    case 2: p = &d->ext_omega; break;
    case 3: p = &d->ext_omega_inv; break;
    case 4: p = &d->g_coset; break;
    case 5: p = &d->g_coset_inv; break;
    case 6: p = &d->ifft_divisor; break;
    case 7: p = &d->ext_ifft_divisor; break;
    default:
        if (which >= 8 && (uint32_t)(which - 8) < d->nt) p = &d->t_eval[which - 8];
    }
    if (!p) return failf(H2V_EINVAL, "domain_constant: index %d out of range", which);
    fe_to_u64x4(*p, out);
    return H2V_OK;
}

// ---- the scalar / index helpers of poly/domain.rs (SURVEY.md 8(a) row a12); host-side, no device work
// EvaluationDomain::rotate_omega(value, rotation) = value * omega^rotation
int h2v_domain_rotate_omega(h2v_domain_t h, const uint64_t value[4], int32_t rotation, uint64_t out[4]) {
    if (!h || !value || !out) return failf(H2V_EINVAL, "rotate_omega: NULL argument");
    const DomRep *d = h->rep[0];
    fe w = rotation >= 0 ? fe_pow_u64<Fr>(d->omega, (uint64_t)rotation) : fe_pow_u64<Fr>(d->omega_inv, (uint64_t)(-(int64_t)rotation));
    fe_to_u64x4(fe_mul<Fr>(fe_from_u64x4(value), w), out);
    return H2V_OK;
}
// EvaluationDomain::rotate_extended(poly, rotation): cyclic shift of an extended-domain column by
// rotation * 2^(extended_k - k) positions (out[i] = in[i + shift]); in != out
int h2v_domain_rotate_extended(h2v_domain_t h, const uint64_t *in, int32_t rotation, uint64_t *out) {
    if (!h || !in || !out || in == out) return failf(H2V_EINVAL, "rotate_extended: NULL or aliased buffers");
    const DomRep *d = h->rep[0];
    const size_t en = (size_t)1 << d->ek;
    const uint64_t per = (uint64_t)1 << (d->ek - d->k);
    const uint64_t mag = (uint64_t)(rotation < 0 ? -(int64_t)rotation : (int64_t)rotation) * per % en;
    const size_t sh = (size_t)(rotation >= 0 ? mag : (en - mag) % en);     // rotate_left(mag) / rotate_right(mag)
    memcpy(out, in + 4 * sh, (en - sh) * 32);
    memcpy(out + 4 * (en - sh), in, sh * 32);
    return H2V_OK;
}
// EvaluationDomain::l_i_range(x, xn, rotations): out[t] = l_i(x) for i = rot_lo + t, rot_lo <= i < rot_hi, where
// l_i(x) = omega^i (x^n - 1) / (n (x - omega^i)); xn = x^n is supplied as upstream's callers do.
int h2v_domain_l_i_range(h2v_domain_t h, const uint64_t x[4], const uint64_t xn[4], int32_t rot_lo, int32_t rot_hi, uint64_t *out) {
    if (!h || !x || !xn || (rot_hi > rot_lo && !out)) return failf(H2V_EINVAL, "l_i_range: NULL argument");
    const DomRep *d = h->rep[0];
    if (rot_hi < rot_lo || (int64_t)rot_hi - rot_lo > (1 << 24)) return failf(H2V_EINVAL, "l_i_range: bad rotation range");
    const fe X = fe_from_u64x4(x), one = fe_one<Fr>();
    const fe common = fe_mul<Fr>(fe_sub<Fr>(fe_from_u64x4(xn), one), d->ifft_divisor);    // barycentric_weight = 1 / n
    const size_t cnt = (size_t)((int64_t)rot_hi - rot_lo);
    std::vector<fe> w(cnt), den(cnt), pre(cnt);
    fe cur = rot_lo >= 0 ? fe_pow_u64<Fr>(d->omega, (uint64_t)rot_lo) : fe_pow_u64<Fr>(d->omega_inv, (uint64_t)(-(int64_t)rot_lo));
    for (size_t t = 0; t < cnt; ++t) {
        w[t] = cur;
        den[t] = fe_sub<Fr>(X, cur);
        cur = fe_mul<Fr>(cur, d->omega);
    }
    // batch_invert (zeros skipped, as ff::BatchInvert does: x on the domain gives l_i(x) = 0 there, like upstream)
    fe acc = one;
    for (size_t t = 0; t < cnt; ++t) {
        pre[t] = acc;
        if (!fe_is_zero(den[t])) acc = fe_mul<Fr>(acc, den[t]);
    }
    fe inv = fe_inv<Fr>(acc);
    for (size_t t = cnt; t-- > 0;) {
        fe r = fe_zero();
        if (!fe_is_zero(den[t])) {
            r = fe_mul<Fr>(inv, pre[t]);
            inv = fe_mul<Fr>(inv, den[t]);
        }
        fe_to_u64x4(fe_mul<Fr>(fe_mul<Fr>(r, common), w[t]), out + 4 * t);
    }
    return H2V_OK;
}
// EvaluationDomain::{empty_coeff, empty_lagrange, empty_extended, constant_lagrange, constant_extended}: a column of
// the basis' length filled with `scalar` (NULL = zero).  basis: 0 coeff, 1 lagrange (both 2^k), 2 extended (2^extended_k)
int h2v_domain_fill(h2v_domain_t h, int basis, const uint64_t scalar[4], uint64_t *out) {
    if (!h || !out) return failf(H2V_EINVAL, "domain_fill: NULL argument");
    const DomRep *d = h->rep[0];
    if (basis < 0 || basis > 2) return failf(H2V_EINVAL, "domain_fill: basis must be 0, 1 or 2");
    const size_t len = (size_t)1 << (basis == 2 ? d->ek : d->k);
    if (!scalar) {
        memset(out, 0, len * 32);
    } else {
        for (size_t i = 0; i < len; ++i) memcpy(out + 4 * i, scalar, 32);
    }
    return H2V_OK;
}

static int rep_domain_transform_dev(DomRep *d, int op, const void *d_in, size_t in_stride, void *d_out, size_t out_stride,
                             size_t n_cols) {
    if (!d) return failf(H2V_EINVAL, "transform: NULL domain");
    if (n_cols && (!d_in || !d_out)) return failf(H2V_EINVAL, "transform: NULL buffer");
    if (op < 0 || op > H2V_OP_DIVIDE_BY_VANISHING) return failf(H2V_EINVAL, "unknown domain op %d", op);
    // the output column doubles as the work buffer of the in-place passes: it needs the full transform size
    const size_t work_len = (size_t)1 << (op >= H2V_OP_COEFF_TO_EXTENDED ? d->ek : d->k);
    if (in_stride < op_in_len(d, op) || out_stride < work_len)
        return failf(H2V_EINVAL, "transform: stride shorter than the column (out_stride must cover 2^%s)",
                    op >= H2V_OP_COEFF_TO_EXTENDED ? "extended_k" : "k");
    H2V_TRY(use_device(d->dev));
    return sync_call(d->mu, d->stream, 7, "transform", [&](Timer &) {
        return domain_op_dev(d, d->stream, op, (const fe *)d_in, in_stride, (fe *)d_out, out_stride, n_cols);
    });
}

static int rep_domain_transform_batch(DomRep *d, int op, const uint64_t *const *in, uint64_t *const *out, size_t n_cols) {
    if (!d) return failf(H2V_EINVAL, "transform: NULL domain");
    if (op < 0 || op > H2V_OP_DIVIDE_BY_VANISHING) return failf(H2V_EINVAL, "unknown domain op %d", op);
    if (n_cols == 0) return H2V_OK;
    if (!in || !out) return failf(H2V_EINVAL, "transform: NULL buffer");
    int rc = use_device(d->dev);
    if (rc) return rc;
    const size_t nin = op_in_len(d, op), nout = op_out_len(d, op);
    const size_t out_stride = std::max(nout, (size_t)1 << (op >= H2V_OP_COEFF_TO_EXTENDED ? d->ek : d->k));
    if (n_cols * out_stride * sizeof(fe) <= ((size_t)8 << 20)) {
        DomRep::Lane *ln = lock_lane(d);
        std::lock_guard<std::mutex> lk(ln->mu, std::adopt_lock);
        if (!ln->st) H2V_CU(cudaStreamCreateWithFlags(&ln->st, cudaStreamNonBlocking));
        if ((rc = ln->stage_a.ensure(n_cols * nin * sizeof(fe)))) return rc;
        if ((rc = ln->stage_b.ensure(n_cols * out_stride * sizeof(fe)))) return rc;
        for (size_t c = 0; c < n_cols; ++c) {
            if (!in[c] || !out[c]) {
                cudaStreamSynchronize(ln->st);
                return failf(H2V_EINVAL, "transform: column %zu is NULL", c);
            }
        }
        H2V_CU(stage_columns(true, ln->stage_a.as<fe>(), nin, in, n_cols, nin, ln->st));
        rc = domain_op_dev(d, ln->st, op, ln->stage_a.as<fe>(), nin, ln->stage_b.as<fe>(), out_stride, n_cols);
        if (rc) {
            cudaStreamSynchronize(ln->st);
            return rc;
        }
        H2V_CU(stage_columns(false, ln->stage_b.as<fe>(), out_stride, out, n_cols, nout, ln->st));
        H2V_CU(cudaStreamSynchronize(ln->st));
        return H2V_OK;
    }
    // Pipelined batch: sub-batches rotate over three pipelines (stream + staging each) with no sync in between, so the
    // upload of sub-batch i+1, the kernels of sub-batch i and the download of sub-batch i-1 overlap -- PCIe is full
    // duplex and the transforms are several times faster than the link, so the call runs at the slower direction's rate.
    // Sub-batch size: at least ~6 per call (to fill the pipeline), 4..64 MB of output each.
    std::lock_guard<std::mutex> lk(d->mu);
    const size_t col_bytes = out_stride * sizeof(fe);
    size_t per = (n_cols + 5) / 6;
    per = std::max(per, std::max<size_t>(1, ((size_t)4 << 20) / col_bytes));
    per = std::min(per, std::max<size_t>(1, ((size_t)64 << 20) / col_bytes));
    per = std::min(per, n_cols);
    const int NP = 3;
    if (!d->pipe_stream) {
        H2V_CU(cudaStreamCreateWithFlags(&d->pipe_stream, cudaStreamNonBlocking));
        H2V_CU(cudaStreamCreateWithFlags(&d->pipe_stream2, cudaStreamNonBlocking));
    }
    cudaStream_t pst[NP] = {d->stream, d->pipe_stream, d->pipe_stream2};
    DevBuf *pa[NP] = {&d->stage_a, &d->pipe_a, &d->pipe_a2}, *pb[NP] = {&d->stage_b, &d->pipe_b, &d->pipe_b2};
    auto sync_all = [&] {
        for (int b = 0; b < NP; ++b) cudaStreamSynchronize(pst[b]);
    };
    for (int b = 0; b < NP; ++b) {
        if ((rc = pa[b]->ensure(per * nin * sizeof(fe)))) return rc;
        if ((rc = pb[b]->ensure(per * out_stride * sizeof(fe)))) return rc;
    }
    size_t it = 0;
    for (size_t c0 = 0; c0 < n_cols; c0 += per, ++it) {
        const size_t cols = std::min(per, n_cols - c0);
        const int b = (int)(it % NP);
        for (size_t c = 0; c < cols; ++c) {
            if (!in[c0 + c] || !out[c0 + c]) {
                sync_all();
                return failf(H2V_EINVAL, "transform: column %zu is NULL", c0 + c);
            }
        }
        {
            cudaError_t e = stage_columns(true, pa[b]->as<fe>(), nin, in + c0, cols, nin, pst[b]);
            if (e != cudaSuccess) {
                sync_all();
                return failf(H2V_ECUDA, "transform: upload failed: %s", cudaGetErrorString(e));
            }
        }
        rc = domain_op_dev(d, pst[b], op, pa[b]->as<fe>(), nin, pb[b]->as<fe>(), out_stride, cols);
        if (rc) {
            sync_all();
            return rc;
        }
        {
            cudaError_t e = stage_columns(false, pb[b]->as<fe>(), out_stride, out + c0, cols, nout, pst[b]);
            if (e != cudaSuccess) {
                sync_all();
                return failf(H2V_ECUDA, "transform: download failed: %s", cudaGetErrorString(e));
            }
        }
    }
    for (int b = 0; b < NP; ++b) H2V_CU(cudaStreamSynchronize(pst[b]));
    return H2V_OK;
}
// one host column on the primary replica
static int one_col(h2v_domain_t h, int op, const uint64_t *in, uint64_t *out) {
    DomRep *d = dom_rep(h, nullptr);
    return d ? rep_domain_transform_batch(d, op, &in, &out, 1) : H2V_EINVAL;
}
int h2v_lagrange_to_coeff(h2v_domain_t h, uint64_t *a) { return one_col(h, H2V_OP_LAGRANGE_TO_COEFF, a, a); }
int h2v_coeff_to_lagrange(h2v_domain_t h, uint64_t *a) { return one_col(h, H2V_OP_COEFF_TO_LAGRANGE, a, a); }
int h2v_coeff_to_extended(h2v_domain_t h, const uint64_t *in, uint64_t *out) { return one_col(h, H2V_OP_COEFF_TO_EXTENDED, in, out); }
int h2v_extended_to_coeff(h2v_domain_t h, const uint64_t *in, uint64_t *out) { return one_col(h, H2V_OP_EXTENDED_TO_COEFF, in, out); }
int h2v_divide_by_vanishing_poly(h2v_domain_t h, uint64_t *a) {
    DomRep *d = dom_rep(h, nullptr);
    if (!d) return H2V_EINVAL;
    if (!a) return failf(H2V_EINVAL, "divide_by_vanishing_poly: NULL argument");
    int rc = use_device(d->dev);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(d->mu);
    size_t en = (size_t)1 << d->ek;
    if ((rc = d->stage_b.ensure(en * sizeof(fe)))) return rc;
    H2V_CU(cudaMemcpyAsync(d->stage_b.p, a, en * sizeof(fe), cudaMemcpyHostToDevice, d->stream));
    fr_scale_mod_kernel<<<dim3((unsigned)((en + 255) / 256), 1), 256, 0, d->stream>>>(d->stage_b.as<fe>(), en, d->dconst.as<fe>() + 8, d->nt,
                                                                                     (uint32_t)en);
    H2V_LAUNCHED();
    H2V_CU(cudaMemcpyAsync(a, d->stage_b.p, en * sizeof(fe), cudaMemcpyDeviceToHost, d->stream));
    H2V_CU(cudaStreamSynchronize(d->stream));
    return H2V_OK;
}

}  // extern "C"

// ================================================================== polynomial primitives ("next" row 2)
namespace {
// the calling thread on device `dev`, *P <- the polynomial context there
int poly_on(int dev, PolyCtx **P) {
    DevCtx *cx;
    H2V_TRY(use_device(dev, &cx));
    *P = &cx->poly;
    return H2V_OK;
}
int poly_ctx_ready(PolyCtx *P) {      // P->mu held
    if (!P->st) H2V_CU(cudaStreamCreateWithFlags(&P->st, cudaStreamNonBlocking));
    return H2V_OK;
}
// I[i] = 1 / X[i] for n non-zero elements (one inversion in total); X and I are device arrays
template <class F> int run_batch_invert(cudaStream_t st, const fe *X, fe *I, uint32_t n, DevBuf &scratch) {
    const uint32_t G = 16;
    uint32_t sizes[16], levels = 0;
    size_t total = 0;
    for (uint64_t v = n;;) {
        sizes[levels++] = (uint32_t)v;
        if (v <= 1 || levels >= 16) break;
        v = (v + G - 1) / G;
        total += v;
    }
    if (sizes[levels - 1] != 1) return failf(H2V_EINVAL, "batch_invert: n = %u unsupported", n);
    // scratch: X_l (levels >= 1), P_l (all levels), I_l (levels >= 1)
    int rc = scratch.ensure((2 * total + n + total + 16) * sizeof(fe));
    if (rc) return rc;
    fe *base = scratch.as<fe>();
    const fe *Xl[16];
    fe *Xw[16], *Pl[16], *Il[16];
    Xl[0] = X;
    Il[0] = I;
    fe *cur = base;
    Pl[0] = cur;
    cur += n;
    for (uint32_t l = 1; l < levels; ++l) {
        Xw[l] = cur; cur += sizes[l];
        Pl[l] = cur; cur += sizes[l];
        Il[l] = cur; cur += sizes[l];
        Xl[l] = Xw[l];
    }
    for (uint32_t l = 0; l + 1 < levels; ++l) {
        binv_up_kernel<F><<<(sizes[l + 1] + 127) / 128, 128, 0, st>>>(Xl[l], Pl[l], Xw[l + 1], sizes[l], G);
        H2V_LAUNCHED();
    }
    binv_top_kernel<F><<<1, 32, 0, st>>>(Xl[levels - 1], Il[levels - 1]);
    H2V_LAUNCHED();
    for (uint32_t l = levels - 1; l-- > 0;) {
        binv_down_kernel<F><<<(sizes[l + 1] + 127) / 128, 128, 0, st>>>(Xl[l], Pl[l], Il[l + 1], Il[l], sizes[l], G);
        H2V_LAUNCHED();
    }
    return H2V_OK;
}
}  // namespace

extern "C" {
int h2v_eval_polynomial_dev(const void *d_polys, size_t stride, size_t n_polys, size_t len, const void *d_points, size_t n_points,
                            void *d_out) {
    if (!n_polys || !n_points) return H2V_OK;
    if (!d_polys || !d_points || !d_out) return failf(H2V_EINVAL, "eval_polynomial: NULL buffer");
    if (n_polys > 65535 || n_points > (1u << 20) || len >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "eval_polynomial: batch too large");
    PolyCtx *P;
    H2V_TRY(poly_on(device_of(d_polys), &P));
    return sync_call(P->mu, P->st, 7, "eval_polynomial", [&](Timer &) {
        poly_eval_kernel<<<dim3((unsigned)n_points, (unsigned)n_polys), 256, 0, P->st>>>((const fe *)d_polys, stride, (uint32_t)len,
                                                                                           (const fe *)d_points, (uint32_t)n_points, (fe *)d_out);
        H2V_LAUNCHED();
        return H2V_OK;
    });
}
int h2v_eval_polynomial_batch(const uint64_t *const *polys, size_t n_polys, size_t len, const uint64_t *points, size_t n_points,
                              uint64_t *out) {
    if (!n_polys || !n_points) return H2V_OK;
    if (!polys || !points || !out) return failf(H2V_EINVAL, "eval_polynomial: NULL buffer");
    if (n_points > (1u << 20) || len >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "eval_polynomial: batch too large");
    PolyCtx *P;
    int rc = poly_on(g_devs[0], &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    cudaStream_t st = P->st;
    const size_t stride = std::max<size_t>(len, 1);
    size_t per = std::max<size_t>(1, ((size_t)1 << 30) / (stride * sizeof(fe)));
    per = std::min<size_t>(std::min(per, n_polys), 65535);
    if ((rc = P->a.ensure(per * stride * sizeof(fe))) || (rc = P->b.ensure(n_points * sizeof(fe))) ||
        (rc = P->c.ensure(per * n_points * sizeof(fe))))
        return rc;
    H2V_CU(cudaMemcpyAsync(P->b.p, points, n_points * sizeof(fe), cudaMemcpyHostToDevice, st));
    for (size_t c0 = 0; c0 < n_polys; c0 += per) {
        size_t cols = std::min(per, n_polys - c0);
        for (size_t c = 0; c < cols; ++c) {
            if (!polys[c0 + c] && len) return failf(H2V_EINVAL, "eval_polynomial: polys[%zu] is NULL", c0 + c);
            if (len) H2V_CU(cudaMemcpyAsync(P->a.as<fe>() + c * stride, polys[c0 + c], len * sizeof(fe), cudaMemcpyHostToDevice, st));
        }
        poly_eval_kernel<<<dim3((unsigned)n_points, (unsigned)cols), 256, 0, st>>>(P->a.as<fe>(), stride, (uint32_t)len, P->b.as<fe>(),
                                                                                  (uint32_t)n_points, P->c.as<fe>());
        H2V_LAUNCHED();
        H2V_CU(cudaMemcpyAsync(out + 4 * c0 * n_points, P->c.p, cols * n_points * sizeof(fe), cudaMemcpyDeviceToHost, st));
        H2V_CU(cudaStreamSynchronize(st));
    }
    return H2V_OK;
}
int h2v_batch_invert(uint64_t *a, size_t n) {
    if (!n) return H2V_OK;
    if (!a) return failf(H2V_EINVAL, "batch_invert: NULL buffer");
    if (n >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "batch_invert: n too large");
    PolyCtx *P;
    int rc = poly_on(g_devs[0], &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    cudaStream_t st = P->st;
    if ((rc = P->a.ensure(n * sizeof(fe))) || (rc = P->b.ensure(n * sizeof(fe))) || (rc = P->c.ensure(n * sizeof(fe)))) return rc;
    H2V_CU(cudaMemcpyAsync(P->a.p, a, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    const unsigned gb = (unsigned)((n + 255) / 256);
    fr_zero_to_one_kernel<<<gb, 256, 0, st>>>(P->a.as<fe>(), P->b.as<fe>(), (uint32_t)n);
    H2V_LAUNCHED();
    if ((rc = run_batch_invert<FrP>(st, P->b.as<fe>(), P->c.as<fe>(), (uint32_t)n, P->tree))) return rc;
    fr_select_inverse_kernel<<<gb, 256, 0, st>>>(P->a.as<fe>(), P->c.as<fe>(), P->b.as<fe>(), (uint32_t)n);
    H2V_LAUNCHED();
    H2V_CU(cudaMemcpyAsync(a, P->b.p, n * sizeof(fe), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}
// out[c][0] = 1, out[c][i+1] = out[c][i] * num[c][i] / den[c][i] for `cols` contiguous columns of n elements (device)
static int run_grand_product(PolyCtx *P, const fe *num, const fe *den, uint32_t n, uint32_t cols, fe *out) {
    int rc;
    const cudaStream_t st = P->st;
    const uint32_t ntiles = (n + H2V_FR_TILE - 1) / H2V_FR_TILE;
    const size_t tot = (size_t)n * cols;
    if ((rc = P->c.ensure(tot * sizeof(fe))) || (rc = P->e.ensure(tot * sizeof(fe))) ||
        (rc = P->d.ensure(((size_t)ntiles * cols + 1) * sizeof(fe))))
        return rc;
    // One inversion for all columns, with the semantics of ff `BatchInvert::batch_invert` that upstream's permutation and
    // lookup provers call: a zero denominator is skipped (its "inverse" stays 0, the running product is 0 from there on)
    // and does not disturb any other element of the batch.
    const unsigned gt = (unsigned)((tot + 255) / 256);
    fr_zero_to_one_kernel<<<gt, 256, 0, st>>>(den, P->e.as<fe>(), (uint32_t)tot);
    H2V_LAUNCHED();
    if ((rc = run_batch_invert<FrP>(st, P->e.as<fe>(), P->c.as<fe>(), (uint32_t)tot, P->tree))) return rc;
    fr_select_inverse_kernel<<<gt, 256, 0, st>>>(den, P->c.as<fe>(), P->e.as<fe>(), (uint32_t)tot);
    H2V_LAUNCHED();
    fr_prod_tiles_kernel<<<dim3(ntiles, cols), 256, 0, st>>>(num, P->e.as<fe>(), n, P->d.as<fe>());
    H2V_LAUNCHED();
    fr_scan_top_kernel<OpMul><<<dim3(1, cols), 256, 0, st>>>(P->d.as<fe>(), ntiles);
    H2V_LAUNCHED();
    fr_prod_apply_kernel<<<dim3(ntiles, cols), 256, 0, st>>>(num, P->e.as<fe>(), n, P->d.as<fe>(), out);
    H2V_LAUNCHED();
    return H2V_OK;
}
int h2v_grand_product(const uint64_t *num, const uint64_t *den, size_t n, uint64_t *out) {
    if (!n) return H2V_OK;
    if (!num || !den || !out) return failf(H2V_EINVAL, "grand_product: NULL buffer");
    if (n >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "grand_product: n too large");
    PolyCtx *P;
    int rc = poly_on(g_devs[0], &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    cudaStream_t st = P->st;
    if ((rc = P->a.ensure(n * sizeof(fe))) || (rc = P->b.ensure(n * sizeof(fe)))) return rc;
    H2V_CU(cudaMemcpyAsync(P->a.p, num, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(P->b.p, den, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    // the running product overwrites the staged denominators once their inverses exist
    if ((rc = run_grand_product(P, P->a.as<fe>(), P->b.as<fe>(), (uint32_t)n, 1, P->b.as<fe>()))) {
        cudaStreamSynchronize(st);
        return rc;
    }
    H2V_CU(cudaMemcpyAsync(out, P->b.p, n * sizeof(fe), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}
int h2v_grand_product_dev(const void *d_num, const void *d_den, size_t n, size_t n_cols, void *d_out) {
    if (!n || !n_cols) return H2V_OK;
    if (!d_num || !d_den || !d_out) return failf(H2V_EINVAL, "grand_product: NULL buffer");
    if (n_cols > 65535 || n * n_cols >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "grand_product: batch too large");
    PolyCtx *P;
    H2V_TRY(poly_on(device_of(d_num), &P));
    return sync_call(P->mu, P->st, 7, "grand_product", [&](Timer &) {
        return run_grand_product(P, (const fe *)d_num, (const fe *)d_den, (uint32_t)n, (uint32_t)n_cols, (fe *)d_out);
    });
}
// every job's division in one set of launches (poly.cuh KateCol); a, q device-resident (q: n - 1 coefficients, must not
// overlap a); P->mu held by the caller
static int run_kate_division(PolyCtx *P, const KateJob *jobs, size_t n_jobs) {
    int rc;
    const cudaStream_t st = P->st;
    std::vector<KateCol> cols;
    uint32_t nmax = 0;
    for (size_t j = 0; j < n_jobs; ++j) {
        if (jobs[j].n <= 1) continue;
        KateCol c;
        c.a = (const fe *)jobs[j].a;
        c.q = (fe *)jobs[j].q;
        c.n = (uint32_t)jobs[j].n;
        c.b = fe_from_u64x4(jobs[j].b);
        c.binv = fe_is_zero(c.b) ? fe_zero() : fe_inv<Fr>(c.b);      // one host-side inversion per point
        cols.push_back(c);
        nmax = std::max(nmax, c.n);
    }
    if (cols.empty()) return H2V_OK;
    if (cols.size() > 65535) return failf(H2V_EINVAL, "kate_division: %zu columns in one call", cols.size());
    const uint32_t ntiles = (nmax + H2V_FR_TILE - 1) / H2V_FR_TILE;
    if ((rc = P->d.ensure((cols.size() * ntiles + 1) * sizeof(fe))) || (rc = P->e.ensure(cols.size() * sizeof(KateCol)))) return rc;
    H2V_CU(cudaMemcpyAsync(P->e.p, cols.data(), cols.size() * sizeof(KateCol), cudaMemcpyHostToDevice, st));
    const KateCol *d_cols = P->e.as<KateCol>();
    fe *tile = P->d.as<fe>();
    const dim3 grid(ntiles, (unsigned)cols.size());
    kate_tiles_kernel<<<grid, 256, 0, st>>>(d_cols, tile, ntiles);
    H2V_LAUNCHED();
    fr_scan_top_kernel<OpAdd><<<dim3(1, (unsigned)cols.size()), 256, 0, st>>>(tile, ntiles);
    H2V_LAUNCHED();
    kate_apply_kernel<<<grid, 256, 0, st>>>(d_cols, tile, ntiles);
    H2V_LAUNCHED();
    return H2V_OK;
}
}  // extern "C"
namespace h2v {
int kate_division_batch_dev(const KateJob *jobs, size_t n_jobs) {
    if (!n_jobs) return H2V_OK;
    if (!jobs) return failf(H2V_EINVAL, "kate_division: NULL job list");
    for (size_t j = 0; j < n_jobs; ++j) {
        if (jobs[j].n <= 1) continue;
        if (!jobs[j].a || !jobs[j].q) return failf(H2V_EINVAL, "kate_division: NULL buffer");
        if (jobs[j].n >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "kate_division: n too large");
    }
    PolyCtx *P;
    int rc = poly_on(device_of(jobs[0].a), &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    rc = run_kate_division(P, jobs, n_jobs);
    cudaError_t e = cudaStreamSynchronize(P->st);
    if (rc) return rc;
    if (e != cudaSuccess) return failf(H2V_ECUDA, "kate_division: %s", cudaGetErrorString(e));
    return H2V_OK;
}
}  // namespace h2v
extern "C" {
int h2v_kate_division_dev(const void *d_a, size_t n, const uint64_t b[4], void *d_out) {
    if (n <= 1) return H2V_OK;
    if (!d_a || !b || !d_out) return failf(H2V_EINVAL, "kate_division: NULL buffer");
    KateJob job{d_a, d_out, n, {b[0], b[1], b[2], b[3]}};
    return kate_division_batch_dev(&job, 1);
}
int h2v_kate_division(const uint64_t *a, size_t n, const uint64_t b[4], uint64_t *out) {
    if (n <= 1) return H2V_OK;
    if (!a || !b || !out) return failf(H2V_EINVAL, "kate_division: NULL buffer");
    if (n >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "kate_division: n too large");
    PolyCtx *P;
    int rc = poly_on(g_devs[0], &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    cudaStream_t st = P->st;
    if ((rc = P->a.ensure(n * sizeof(fe))) || (rc = P->b.ensure(n * sizeof(fe)))) return rc;
    H2V_CU(cudaMemcpyAsync(P->a.p, a, n * sizeof(fe), cudaMemcpyHostToDevice, st));
    const KateJob job{P->a.p, P->b.p, n, {b[0], b[1], b[2], b[3]}};
    if ((rc = run_kate_division(P, &job, 1))) {
        cudaStreamSynchronize(st);
        return rc;
    }
    H2V_CU(cudaMemcpyAsync(out, P->b.p, (n - 1) * sizeof(fe), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}
}  // extern "C"

// ================================================================== lookup argument: permuted columns
namespace h2v {
int sort_canonical_dev(cudaStream_t st, const fe *const *d_srcs, uint32_t slices, uint32_t u, uint32_t n_pad, fe *keys) {
    lookup_canon_pad_batch_kernel<<<dim3((n_pad + 255) / 256, slices), 256, 0, st>>>(d_srcs, keys, u, n_pad);
    H2V_LAUNCHED();
    const uint32_t tile = std::min<uint32_t>(H2V_SORT_TILE, n_pad);
    const unsigned tiles_n = n_pad / tile;
    const size_t smem = (size_t)tile * sizeof(fe);
    bitonic_tile_kernel<<<dim3(tiles_n, slices), H2V_SORT_TILE / 2, smem, st>>>(keys, n_pad, 0, 1);
    H2V_LAUNCHED();
    for (uint32_t k = 2 * tile; k <= n_pad && k; k <<= 1) {
        for (uint32_t j = k >> 1; j >= tile; j >>= 1) {
            bitonic_global_kernel<<<dim3((n_pad / 2 + 255) / 256, slices), 256, 0, st>>>(keys, n_pad, k, j);
            H2V_LAUNCHED();
        }
        bitonic_tile_kernel<<<dim3(tiles_n, slices), H2V_SORT_TILE / 2, smem, st>>>(keys, n_pad, k, 0);
        H2V_LAUNCHED();
    }
    return H2V_OK;
}
int scan_u32_dev(cudaStream_t st, const uint32_t *cnt, uint32_t len, uint32_t *offs, uint32_t *tiles, uint32_t *scratch, uint32_t *total) {
    const uint32_t ntiles = (len + H2V_SCAN_TILE - 1) / H2V_SCAN_TILE;
    msm_scan_tiles_kernel<<<ntiles, 256, 0, st>>>(cnt, tiles, len);
    H2V_LAUNCHED();
    msm_scan_top_kernel<<<1, 256, 0, st>>>(tiles, ntiles, total);
    H2V_LAUNCHED();
    msm_scan_apply_kernel<<<ntiles, 256, 0, st>>>(cnt, tiles, offs, scratch, len);
    H2V_LAUNCHED();
    return H2V_OK;
}
}  // namespace h2v
namespace {
// A', S' of `u` usable rows from device-resident input / table expressions (Montgomery); P->mu held by the caller
// All lookup arguments of one proof phase in one set of launches (lookup.cuh): inputs[l] / tables[l] are device columns,
// the permuted columns land at out_a + l * a_stride / out_s + l * s_stride.  Identical table pointers are sorted once.
int run_permute_batch(PolyCtx *P, const fe *const *inputs, const fe *const *tables, uint32_t L, uint32_t u, fe *d_out_a, size_t a_stride,
                      fe *d_out_s, size_t s_stride) {
    int rc;
    const cudaStream_t st = P->st;
    uint32_t n_pad = 1;
    while (n_pad < u) n_pad <<= 1;
    std::vector<const fe *> srcs(inputs, inputs + L);
    std::vector<uint32_t> tmap(L);
    for (uint32_t l = 0; l < L; ++l) {
        uint32_t t = L;
        for (; t < srcs.size(); ++t)
            if (srcs[t] == tables[l]) break;
        if (t == srcs.size()) srcs.push_back(tables[l]);
        tmap[l] = t;
    }
    const uint32_t slices = (uint32_t)srcs.size();
    const size_t rows = (size_t)L * u;
    if (rows >= ((size_t)1 << 31)) return failf(H2V_EINVAL, "permute_expression_pair: batch too large");
    const uint32_t ntiles = (uint32_t)((rows + H2V_SCAN_TILE - 1) / H2V_SCAN_TILE);
    const size_t ptr_words = ((size_t)slices * sizeof(void *) + 3) / 4;
    if ((rc = P->a.ensure((size_t)slices * n_pad * sizeof(fe))) ||
        (rc = P->tree.ensure((6 * rows + 2 * ntiles + 16 + L + ptr_words + 8) * sizeof(uint32_t))))
        return rc;
    fe *keys = P->a.as<fe>();
    uint32_t *rep = P->tree.as<uint32_t>(), *free_ = rep + rows, *rep_offs = free_ + rows, *free_offs = rep_offs + rows;
    uint32_t *scratch = free_offs + rows, *rep_rows = scratch + rows, *tiles = rep_rows + rows, *totals = tiles + 2 * ntiles;
    int *err = reinterpret_cast<int *>(totals + 2);
    uint32_t *d_tmap = totals + 4;
    uintptr_t pa = reinterpret_cast<uintptr_t>(d_tmap + L);
    pa = (pa + 7) & ~(uintptr_t)7;
    const fe **d_srcs = reinterpret_cast<const fe **>(pa);
    H2V_CU(cudaMemsetAsync(err, 0, sizeof(int), st));
    H2V_CU(cudaMemcpyAsync(d_tmap, tmap.data(), L * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(d_srcs, srcs.data(), slices * sizeof(void *), cudaMemcpyHostToDevice, st));
    const unsigned gu = (u + 255) / 256;
    H2V_TRY(sort_canonical_dev(st, d_srcs, slices, u, n_pad, keys));
    lookup_fill_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(free_, 1u, (uint32_t)rows);
    H2V_LAUNCHED();
    lookup_flags_batch_kernel<<<dim3(gu, L), 256, 0, st>>>(keys, d_tmap, u, n_pad, rep, free_, err);
    H2V_LAUNCHED();
    for (int which = 0; which < 2; ++which)
        H2V_TRY(scan_u32_dev(st, which ? free_ : rep, (uint32_t)rows, which ? free_offs : rep_offs, tiles + which * ntiles, scratch, totals + which));
    lookup_emit_input_batch_kernel<<<dim3(gu, L), 256, 0, st>>>(keys, u, n_pad, rep, rep_offs, rep_rows, d_out_a, a_stride, d_out_s, s_stride);
    H2V_LAUNCHED();
    lookup_emit_table_batch_kernel<<<dim3(gu, L), 256, 0, st>>>(keys, d_tmap, L, u, n_pad, free_, free_offs, rep_offs, totals, rep_rows, d_out_s,
                                                                 s_stride, err);
    H2V_LAUNCHED();
    int herr = 0;
    H2V_CU(cudaMemcpyAsync(&herr, err, sizeof(int), cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    if (herr == 1) return failf(H2V_EINVAL, "permute_expression_pair: an input value is not in the table (ConstraintSystemFailure)");
    if (herr) return failf(H2V_ECUDA, "permute_expression_pair: leftover count mismatch");
    return H2V_OK;
}
int run_permute_pair(PolyCtx *P, const fe *d_in_a, const fe *d_in_t, uint32_t u, fe *d_out_a, fe *d_out_s) {
    return run_permute_batch(P, &d_in_a, &d_in_t, 1, u, d_out_a, 0, d_out_s, 0);
}
}  // namespace

extern "C" {
int h2v_permute_expression_pair_dev(const void *d_input, const void *d_table, size_t usable_rows, void *d_permuted_input,
                                    void *d_permuted_table) {
    if (!usable_rows) return H2V_OK;
    if (!d_input || !d_table || !d_permuted_input || !d_permuted_table) return failf(H2V_EINVAL, "permute_expression_pair: NULL buffer");
    if (usable_rows > ((size_t)1 << 28)) return failf(H2V_EINVAL, "permute_expression_pair: too many rows");
    PolyCtx *P;
    H2V_TRY(poly_on(device_of(d_input), &P));
    return sync_call(P->mu, P->st, 7, "permute_expression_pair", [&](Timer &) {
        return run_permute_pair(P, (const fe *)d_input, (const fe *)d_table, (uint32_t)usable_rows, (fe *)d_permuted_input,
                                (fe *)d_permuted_table);
    });
}
int h2v_permute_expression_pair_batch_dev(const void *const *d_inputs, const void *const *d_tables, size_t n_lookups, size_t usable_rows,
                                          void *d_permuted_inputs, size_t input_stride, void *d_permuted_tables, size_t table_stride) {
    if (!usable_rows || !n_lookups) return H2V_OK;
    if (!d_inputs || !d_tables || !d_permuted_inputs || !d_permuted_tables) return failf(H2V_EINVAL, "permute_expression_pair: NULL buffer");
    if (usable_rows > ((size_t)1 << 28) || n_lookups > 65535) return failf(H2V_EINVAL, "permute_expression_pair: too many rows / lookups");
    if (n_lookups > 1 && (input_stride < usable_rows || table_stride < usable_rows))
        return failf(H2V_EINVAL, "permute_expression_pair: output stride shorter than the usable rows");
    for (size_t l = 0; l < n_lookups; ++l)
        if (!d_inputs[l] || !d_tables[l]) return failf(H2V_EINVAL, "permute_expression_pair: lookup %zu has a NULL column", l);
    PolyCtx *P;
    H2V_TRY(poly_on(device_of(d_inputs[0]), &P));
    return sync_call(P->mu, P->st, 7, "permute_expression_pair", [&](Timer &) {
        return run_permute_batch(P, (const fe *const *)d_inputs, (const fe *const *)d_tables, (uint32_t)n_lookups, (uint32_t)usable_rows,
                                 (fe *)d_permuted_inputs, input_stride, (fe *)d_permuted_tables, table_stride);
    });
}
int h2v_permute_expression_pair(const uint64_t *input, const uint64_t *table, size_t usable_rows, uint64_t *permuted_input,
                                uint64_t *permuted_table) {
    if (!usable_rows) return H2V_OK;
    if (!input || !table || !permuted_input || !permuted_table) return failf(H2V_EINVAL, "permute_expression_pair: NULL buffer");
    if (usable_rows > ((size_t)1 << 28)) return failf(H2V_EINVAL, "permute_expression_pair: too many rows");
    PolyCtx *P;
    int rc = poly_on(g_devs[0], &P);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(P->mu);
    if ((rc = poly_ctx_ready(P))) return rc;
    cudaStream_t st = P->st;
    const size_t bytes = usable_rows * sizeof(fe);
    if ((rc = P->c.ensure(bytes)) || (rc = P->d.ensure(bytes))) return rc;
    H2V_CU(cudaMemcpyAsync(P->c.p, input, bytes, cudaMemcpyHostToDevice, st));
    H2V_CU(cudaMemcpyAsync(P->d.p, table, bytes, cudaMemcpyHostToDevice, st));
    // the canonical copies are taken first, so the staging buffers double as the outputs
    if ((rc = run_permute_pair(P, P->c.as<fe>(), P->d.as<fe>(), (uint32_t)usable_rows, P->c.as<fe>(), P->d.as<fe>()))) {
        cudaStreamSynchronize(st);
        return rc;
    }
    H2V_CU(cudaMemcpyAsync(permuted_input, P->c.p, bytes, cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaMemcpyAsync(permuted_table, P->d.p, bytes, cudaMemcpyDeviceToHost, st));
    H2V_CU(cudaStreamSynchronize(st));
    return H2V_OK;
}
}  // extern "C"

// ================================================================== quotient evaluation ("next" row 1)
namespace {
// the replica that holds d_h (made the calling thread's device) and the constants every quotient kernel takes
int quotient_common(h2v_domain_t h, const void *d_h, DomRep **d, QuotientCommon *c) {
    if (!(*d = dom_rep(h, d_h))) return H2V_EINVAL;
    if (!d_h) return failf(H2V_EINVAL, "quotient: NULL buffer");
    c->n_ext = 1u << (*d)->ek;
    c->rot = 1u << ((*d)->ek - (*d)->k);
    return use_device((*d)->dev);
}
// one proof's y, beta, gamma (and `extra_bytes` behind them) into the replica's argument buffer, on its stream: the
// public entry points are groups of one; d->mu held by the caller
int quotient_args(DomRep *d, const uint64_t *y, const uint64_t *beta, const uint64_t *gamma, const void *extra, size_t extra_bytes,
                  QuotientGroup *g, const void **extra_dev) {
    const fe host[3] = {fe_from_u64x4(y), beta ? fe_from_u64x4(beta) : fe_zero(), gamma ? fe_from_u64x4(gamma) : fe_zero()};
    H2V_TRY(d->qargs.ensure(sizeof host + extra_bytes));
    H2V_CU(cudaMemcpyAsync(d->qargs.p, host, sizeof host, cudaMemcpyHostToDevice, d->stream));
    if (extra_bytes)
        H2V_CU(cudaMemcpyAsync((char *)d->qargs.p + sizeof host, extra, extra_bytes, cudaMemcpyHostToDevice, d->stream));
    g->scal = d->qargs.as<fe>();
    if (extra_dev) *extra_dev = (const char *)d->qargs.p + sizeof host;
    return H2V_OK;
}
// the gate columns as strided arrays (ColsStrided) or device tables of column pointers (ColsTable)
template <class Cols> int quotient_gates(h2v_domain_t h, void *d_h, const uint64_t y[4], size_t n_gates, Cols q, Cols a) {
    DomRep *d;
    QuotientCommon c;
    int rc = quotient_common(h, d_h, &d, &c);
    if (rc) return rc;
    if (!y) return failf(H2V_EINVAL, "quotient: NULL buffer");
    if (!n_gates) return H2V_OK;
    if constexpr (std::is_same<Cols, ColsStrided>::value) {
        if (!q.base || !a.base) return failf(H2V_EINVAL, "quotient_gates: NULL buffer");
        if (q.stride < c.n_ext || a.stride < c.n_ext || n_gates > (1u << 20))
            return failf(H2V_EINVAL, "quotient_gates: stride shorter than 2^extended_k, or too many gates");
    } else {
        if (!q.ptrs || !a.ptrs) return failf(H2V_EINVAL, "quotient_gates: NULL pointer table");
        if (n_gates > (1u << 20)) return failf(H2V_EINVAL, "quotient_gates: too many gates");
    }
    return sync_call(d->mu, d->stream, 7, "quotient", [&](Timer &) {
        QuotientGroup g{(fe *)d_h, 0, nullptr};
        H2V_TRY(quotient_args(d, y, nullptr, nullptr, nullptr, 0, &g, nullptr));
        quotient_gates_kernel<<<dim3((c.n_ext + 255) / 256, 1), 256, 0, d->stream>>>(g, c, (uint32_t)n_gates, q, a);
        H2V_LAUNCHED();
        return H2V_OK;
    });
}
// the permutation argument's constants for the sets [set_begin, set_end)
int perm_params(DomRep *d, size_t n_cols, size_t chunk_len, const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last,
                const void *d_l_active, uint32_t blinding_factors, size_t set_begin, size_t set_end, int with_head, QuotientPerm *p) {
    p->delta = fe_pow_u64<Fr>(fr_from_small(7), (uint64_t)1 << 28);   // Fr::DELTA = MULTIPLICATIVE_GENERATOR^(2^S)
    p->g_coset = d->g_coset;
    p->n_cols = (uint32_t)n_cols;
    p->chunk_len = (uint32_t)std::min<size_t>(chunk_len, n_cols);
    p->n_sets = (p->n_cols + p->chunk_len - 1) / p->chunk_len;
    p->last_rot = -(int)(blinding_factors + 1);
    p->z = (const fe *)d_z;
    p->z_stride = z_stride;
    p->z_pstride = 0;
    p->l0 = (const fe *)d_l0; p->l_last = (const fe *)d_l_last; p->l_active = (const fe *)d_l_active;
    if (set_end == (size_t)-1) set_end = p->n_sets;
    if (set_begin > set_end || set_end > p->n_sets)
        return failf(H2V_EINVAL, "quotient_permutation: set range [%zu, %zu) of %u sets", set_begin, set_end, p->n_sets);
    p->set_begin = (uint32_t)set_begin;
    p->set_end = (uint32_t)set_end;
    p->head = with_head ? 1u : 0u;
    p->delta_begin = fe_pow_u64<Fr>(p->delta, (uint64_t)set_begin * p->chunk_len);
    return domain_twiddles(d, 2, &p->tw);
}
}  // namespace

extern "C" {
int h2v_quotient_gates_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], size_t n_gates, const void *d_q, size_t q_stride, const void *d_a,
                           size_t a_stride) {
    return quotient_gates(h, d_h, y, n_gates, ColsStrided{(const fe *)d_q, q_stride, 0}, ColsStrided{(const fe *)d_a, a_stride, 0});
}
int h2v_quotient_gates_ptrs_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], size_t n_gates, const void *const *d_q_ptrs,
                                const void *const *d_a_ptrs) {
    return quotient_gates(h, d_h, y, n_gates, ColsTable{(const fe *const *)d_q_ptrs, 0}, ColsTable{(const fe *const *)d_a_ptrs, 0});
}
static int quotient_permutation_any(h2v_domain_t h, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                    size_t n_cols, size_t chunk_len, const void *d_cols, size_t cols_stride, const void *d_sigma,
                                    size_t sigma_stride, const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last,
                                    const void *d_l_active, uint32_t blinding_factors, bool tables, size_t set_begin = 0,
                                    size_t set_end = (size_t)-1, int with_head = 1) {
    DomRep *d;
    QuotientCommon c;
    int rc = quotient_common(h, d_h, &d, &c);
    if (rc) return rc;
    if (!y) return failf(H2V_EINVAL, "quotient: NULL buffer");
    if (!n_cols) return H2V_OK;   // upstream: `if !sets.is_empty()`
    if (!beta || !gamma || !d_cols || !d_sigma || !d_z || !d_l0 || !d_l_last || !d_l_active)
        return failf(H2V_EINVAL, "quotient_permutation: NULL buffer");
    if (!chunk_len || n_cols > (1u << 20) || blinding_factors + 1 >= (1u << d->k))
        return failf(H2V_EINVAL, "quotient_permutation: chunk_len = 0, too many columns, or blinding_factors >= n - 1");
    if ((!tables && (cols_stride < c.n_ext || sigma_stride < c.n_ext)) || z_stride < c.n_ext)
        return failf(H2V_EINVAL, "quotient_permutation: stride shorter than 2^extended_k");
    QuotientPerm p;
    if ((rc = perm_params(d, n_cols, chunk_len, d_z, z_stride, d_l0, d_l_last, d_l_active, blinding_factors, set_begin, set_end, with_head, &p)))
        return rc;
    return sync_call(d->mu, d->stream, 7, "quotient", [&](Timer &) {
        QuotientGroup g{(fe *)d_h, 0, nullptr};
        H2V_TRY(quotient_args(d, y, beta, gamma, nullptr, 0, &g, nullptr));
        const dim3 grid((c.n_ext + 255) / 256, 1);
        if (tables)
            quotient_permutation_kernel<<<grid, 256, 0, d->stream>>>(g, c, p, ColsTable{(const fe *const *)d_cols, 0},
                                                                    ColsTable{(const fe *const *)d_sigma, 0});
        else
            quotient_permutation_kernel<<<grid, 256, 0, d->stream>>>(g, c, p, ColsStrided{(const fe *)d_cols, cols_stride, 0},
                                                                    ColsStrided{(const fe *)d_sigma, sigma_stride, 0});
        H2V_LAUNCHED();
        return H2V_OK;
    });
}
int h2v_quotient_permutation_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                 size_t n_cols, size_t chunk_len, const void *d_cols, size_t cols_stride, const void *d_sigma,
                                 size_t sigma_stride, const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last,
                                 const void *d_l_active, uint32_t blinding_factors) {
    return quotient_permutation_any(h, d_h, y, beta, gamma, n_cols, chunk_len, d_cols, cols_stride, d_sigma, sigma_stride, d_z, z_stride,
                                    d_l0, d_l_last, d_l_active, blinding_factors, false);
}
int h2v_quotient_permutation_ptrs_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                      size_t n_cols, size_t chunk_len, const void *const *d_col_ptrs, const void *const *d_sigma_ptrs,
                                      const void *d_z, size_t z_stride, const void *d_l0, const void *d_l_last, const void *d_l_active,
                                      uint32_t blinding_factors) {
    return quotient_permutation_any(h, d_h, y, beta, gamma, n_cols, chunk_len, d_col_ptrs, 0, d_sigma_ptrs, 0, d_z, z_stride, d_l0, d_l_last,
                                    d_l_active, blinding_factors, true);
}
int h2v_quotient_permutation_range_ptrs_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                                            size_t n_cols, size_t chunk_len, size_t set_begin, size_t set_end, int with_head,
                                            const void *const *d_col_ptrs, const void *const *d_sigma_ptrs, const void *d_z, size_t z_stride,
                                            const void *d_l0, const void *d_l_last, const void *d_l_active, uint32_t blinding_factors) {
    return quotient_permutation_any(h, d_h, y, beta, gamma, n_cols, chunk_len, d_col_ptrs, 0, d_sigma_ptrs, 0, d_z, z_stride, d_l0, d_l_last,
                                    d_l_active, blinding_factors, true, set_begin, set_end, with_head);
}
int h2v_quotient_lookup_dev(h2v_domain_t h, void *d_h, const uint64_t y[4], const uint64_t beta[4], const uint64_t gamma[4],
                            const void *d_input, const void *d_table, const void *d_perm_input, const void *d_perm_table, const void *d_z,
                            const void *d_l0, const void *d_l_last, const void *d_l_active) {
    DomRep *d;
    QuotientCommon c;
    int rc = quotient_common(h, d_h, &d, &c);
    if (rc) return rc;
    if (!y || !beta || !gamma || !d_input || !d_table || !d_perm_input || !d_perm_table || !d_z || !d_l0 || !d_l_last || !d_l_active)
        return failf(H2V_EINVAL, "quotient_lookup: NULL buffer");
    const void *tab[5] = {d_input, d_table, d_perm_input, d_perm_table, d_z};
    return sync_call(d->mu, d->stream, 7, "quotient", [&](Timer &) {
        QuotientGroup g{(fe *)d_h, 0, nullptr};
        const void *d_tab = nullptr;
        H2V_TRY(quotient_args(d, y, beta, gamma, tab, sizeof tab, &g, &d_tab));
        QuotientLookup p{(const fe *const *)d_tab, 0, 1, (const fe *)d_l0, (const fe *)d_l_last, (const fe *)d_l_active};
        quotient_lookup_kernel<<<dim3((c.n_ext + 255) / 256, 1), 256, 0, d->stream>>>(g, c, p);
        H2V_LAUNCHED();
        return H2V_OK;
    });
}
}  // extern "C"

namespace h2v {
// evaluate_h's three folds for a group of proofs, one launch each (gates, permutation, lookups: upstream's order)
int quotient_batch_dev(h2v_domain_t h, const QuotientBatch &b) {
    DomRep *d;
    QuotientCommon c;
    int rc = quotient_common(h, b.h, &d, &c);
    if (rc) return rc;
    if (!b.n_proofs) return H2V_OK;
    if (!b.scal || b.n_proofs > 65535) return failf(H2V_EINVAL, "quotient: no per-proof scalars, or more than 65535 proofs");
    QuotientPerm p;
    if (b.n_perm) {
        if ((rc = perm_params(d, b.n_perm, b.chunk, b.z, b.z_stride, b.l0, b.l_last, b.l_active, b.blinding_factors, 0, (size_t)-1, 1, &p)))
            return rc;
        p.z_pstride = b.z_pstride;
    }
    return sync_call(d->mu, d->stream, 7, "quotient", [&](Timer &) {
        const QuotientGroup g{(fe *)b.h, b.h_stride, (const fe *)b.scal};
        const dim3 grid((c.n_ext + 255) / 256, (unsigned)b.n_proofs);
        const fe *const *gt = (const fe *const *)b.gate_tab, *const *pt = (const fe *const *)b.perm_tab;
        if (b.n_gates) {
            quotient_gates_kernel<<<grid, 256, 0, d->stream>>>(g, c, (uint32_t)b.n_gates, ColsTable{gt, b.gate_pstride},
                                                              ColsTable{gt + b.n_gates, b.gate_pstride});
            H2V_LAUNCHED();
        }
        if (b.n_perm) {
            quotient_permutation_kernel<<<grid, 256, 0, d->stream>>>(g, c, p, ColsTable{pt, b.perm_pstride}, ColsTable{pt + b.n_perm, b.perm_pstride});
            H2V_LAUNCHED();
        }
        if (b.n_lookups) {
            const QuotientLookup q{(const fe *const *)b.lookup_tab, b.lookup_pstride, (uint32_t)b.n_lookups, (const fe *)b.l0,
                                   (const fe *)b.l_last, (const fe *)b.l_active};
            quotient_lookup_kernel<<<grid, 256, 0, d->stream>>>(g, c, q);
            H2V_LAUNCHED();
        }
        return H2V_OK;
    });
}
}  // namespace h2v

// ================================================================== self-tests
namespace {
template <class F> __global__ void selftest_field_kernel(int op, const fe *a, const fe *b, fe *o, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe x = a[i], y = b ? b[i] : fe_zero(), r;
    if (op == 0) r = fe_mul<F>(x, y);
    else if (op == 1) r = fe_add<F>(x, y);
    else if (op == 2) r = fe_sub<F>(x, y);
    else if (op == 3) r = fe_inv<F>(x);
    else if (op == 4) r = fe_inv_fast<F>(x);
    else if (op == 5) r = fe_sqr<F>(x);                       // dedicated squaring, canonical input
    else if (op == 7) {                                         // Shoup product (Fr only): ANY 256-bit a times the twiddle b (Montgomery)
        r = fe_mul_shoup_lazy<F>(x, fe_from_mont<F>(y), fr_shoup_companion(y));
        fe_reduce_once<F>(r);
    } else {                                                      // op 6: the squaring on a lazily reduced input x + m
        fe m_;
#pragma unroll
        for (int k = 0; k < 8; ++k) m_.v[k] = F::m(k);
        r = fe_sqr_lazy<F>(fe_add_raw(x, m_));
        fe_reduce_once<F>(r);
    }
    o[i] = r;
}
__global__ void selftest_group_kernel(int mode, const affine *p, const affine *q, affine *o, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    xyzz acc = xyzz_from_affine(p[i]);
    if (mode == 0) {
        xyzz_add_mixed(acc, q[i]);
    } else if (mode == 1) {
        // give the second operand a non-trivial ZZ by doubling and adding back: q' = 2q + (-q) = q
        xyzz t = xyzz_from_affine(q[i]);
        t = xyzz_double(t);
        xyzz_add_mixed(t, affine_neg(q[i]));
        xyzz_add(acc, t);
    } else {
        acc = xyzz_double(acc);
    }
    o[i] = xyzz_to_affine(acc);
}
// out[i] = (a*i + b) * G, affine -- synthetic bases with a known discrete log (SURVEY.md 8(d) config 5)
__global__ void __launch_bounds__(128) synthetic_bases_kernel(affine *out, uint64_t a, uint64_t b, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned __int128 k = (unsigned __int128)a * i + b;
    affine g;
    fe c = fe_zero();
    c.v[0] = 1;
    g.x = fe_to_mont<Fq>(c);
    c.v[0] = 2;
    g.y = fe_to_mont<Fq>(c);
    xyzz acc = xyzz_identity();
    for (int bit = 127; bit >= 0; --bit) {
        acc = xyzz_double(acc);
        if ((uint64_t)(k >> bit) & 1) xyzz_add_mixed(acc, g);
    }
    out[i] = xyzz_to_affine(acc);
}
// throughput probes for the building blocks of the hot kernels (registers only, no memory traffic)
template <int ILP> __global__ void __launch_bounds__(256) mul_probe_kernel(fe *out, uint32_t iters) {
    fe x[ILP], y[ILP];
#pragma unroll
    for (int k = 0; k < ILP; ++k) {
        x[k] = fe_one<Fq>();
        y[k] = fe_one<Fq>();
        x[k].v[0] += threadIdx.x + k;
        y[k].v[1] += blockIdx.x + 7 * k;
    }
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < ILP; ++k) x[k] = fe_mul<Fq>(x[k], y[k]);
    }
    fe acc = x[0];
#pragma unroll
    for (int k = 1; k < ILP; ++k) acc = fe_add<Fq>(acc, x[k]);
    if (acc.v[0] == 0x12345678u && acc.v[7] == 0x9abcdef0u) out[0] = acc;
}
__global__ void __launch_bounds__(128, 4) madd_probe_kernel(xyzz *out, uint32_t iters) {
    affine g;
    fe c = fe_zero();
    c.v[0] = 1;
    g.x = fe_to_mont<Fq>(c);
    c.v[0] = 2;
    g.y = fe_to_mont<Fq>(c);
    xyzz acc = xyzz_double_affine(g);
    for (uint32_t k = 0; k < (threadIdx.x & 7); ++k) acc = xyzz_double(acc);
    for (uint32_t it = 0; it < iters; ++it) xyzz_add_mixed(acc, g);
    if (acc.x.v[0] == 0x12345678u && acc.y.v[7] == 0x9abcdef0u) out[0] = acc;
}
// IMAD.WIDE.U32 issue-rate probe.  The multiplicands change every iteration (each chain feeds the
// next one's operand), otherwise ptxas hoists the product and the loop degenerates into IADD3s.
__global__ void __launch_bounds__(256) imad_probe_kernel(uint64_t *out, uint32_t iters, uint32_t seed) {
    uint64_t acc[8];
    uint32_t a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        acc[k] = (uint64_t)(seed + k * 0x9e3779b9u) * (threadIdx.x + 1) + blockIdx.x;
        a[k] = seed * (2 * k + 3) + threadIdx.x;
    }
    uint32_t b = seed | 1u;
    for (uint32_t it = 0; it < iters; ++it) {
        b ^= b << 13;            // xorshift: a non-linear update, so the products cannot be strength-reduced
        b ^= b >> 17;
        b ^= b << 5;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[k]) : "r"(a[k]), "r"(b));
        }
    }
    uint64_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s ^= acc[k];
    if (s == 0x1234567812345678ull) out[0] = s;   // keep the chains alive
}
// A second IMAD.WIDE.U32 issue-rate probe with nothing but multiplier instructions in the loop.  (A plain
// `mad.wide.u32 d, a, b, d` does not qualify: ptxas splits its 64-bit accumulate into IMAD.WIDE + IADD3 + IADD3.X.)
// The loop is made of the carry-chained rows the field code is built from -- mad.lo.cc / madc.hi.cc pairs that ptxas
// fuses into IMAD.WIDE.U32.X -- on four independent 8-limb accumulators; the multiplier of each row is a limb of
// another accumulator, so no product is loop-invariant.  4 wide multiply-adds per row, one ADDC per row besides.
__global__ void __launch_bounds__(256) imad_chain_probe_kernel(uint32_t *out, uint32_t iters, uint32_t seed) {
#ifdef __CUDA_ARCH__      // the row primitives exist in the device pass only
    uint32_t a[4][8], x[8], top = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        x[k] = (seed * (2 * k + 3) + threadIdx.x * 2654435761u) | 1u;
#pragma unroll
        for (int c = 0; c < 4; ++c) a[c][k] = seed + 977u * c + k * 0x9e3779b9u + blockIdx.x;
    }
    for (uint32_t it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            row_mad_top(a[0], x, a[1][2 * r], top);
            row_mad_top(a[1], x, a[2][2 * r], top);
            row_mad_top(a[2], x, a[3][2 * r], top);
            row_mad_top(a[3], x, a[0][2 * r + 1], top);
        }
    }
    uint32_t s = top;
#pragma unroll
    for (int k = 0; k < 8; ++k) s ^= a[0][k] ^ a[1][k] ^ a[2][k] ^ a[3][k];
    if (s == 0x12345678u) out[0] = s;
#endif
}
}  // namespace

extern "C" {
int h2v_selftest_field(int field, int op, const uint64_t *a, const uint64_t *b, size_t n, uint64_t *out) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!a || !out || n == 0) return failf(H2V_EINVAL, "selftest_field: bad argument");
    DevBuf A, B, O;
    if ((rc = A.ensure(n * 32)) || (rc = B.ensure(n * 32)) || (rc = O.ensure(n * 32))) return rc;
    H2V_CU(cudaMemcpy(A.p, a, n * 32, cudaMemcpyHostToDevice));
    if (b) H2V_CU(cudaMemcpy(B.p, b, n * 32, cudaMemcpyHostToDevice));
    unsigned g = (unsigned)((n + 127) / 128);
    if (field == 0) selftest_field_kernel<FrP><<<g, 128>>>(op, A.as<fe>(), b ? B.as<fe>() : nullptr, O.as<fe>(), n);
    else selftest_field_kernel<FqP><<<g, 128>>>(op, A.as<fe>(), b ? B.as<fe>() : nullptr, O.as<fe>(), n);
    H2V_LAUNCHED();
    H2V_CU(cudaDeviceSynchronize());
    H2V_CU(cudaMemcpy(out, O.p, n * 32, cudaMemcpyDeviceToHost));
    A.release(); B.release(); O.release();
    return H2V_OK;
}
int h2v_selftest_group(int mode, const uint64_t *p, const uint64_t *q, size_t n, uint64_t *out_affine) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!p || !q || !out_affine || n == 0) return failf(H2V_EINVAL, "selftest_group: bad argument");
    DevBuf A, B, O;
    if ((rc = A.ensure(n * 64)) || (rc = B.ensure(n * 64)) || (rc = O.ensure(n * 64))) return rc;
    H2V_CU(cudaMemcpy(A.p, p, n * 64, cudaMemcpyHostToDevice));
    H2V_CU(cudaMemcpy(B.p, q, n * 64, cudaMemcpyHostToDevice));
    selftest_group_kernel<<<(unsigned)((n + 63) / 64), 64>>>(mode, A.as<affine>(), B.as<affine>(), O.as<affine>(), n);
    H2V_LAUNCHED();
    H2V_CU(cudaDeviceSynchronize());
    H2V_CU(cudaMemcpy(out_affine, O.p, n * 64, cudaMemcpyDeviceToHost));
    A.release(); B.release(); O.release();
    return H2V_OK;
}
int h2v_srs_setup(uint32_t k, const uint64_t s_mont[4], uint64_t *g_out, uint64_t *g_lagrange_out) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!s_mont || (!g_out && !g_lagrange_out)) return failf(H2V_EINVAL, "srs_setup: NULL argument");
    if (k > 26) return failf(H2V_EINVAL, "srs_setup: k = %u unsupported", k);
    const size_t n = (size_t)1 << k;
    SetupParams sp;
    sp.s = fe_from_u64x4(s_mont);
    sp.n = (uint32_t)n;
    fe root;
    memcpy(root.v, FR_ROOT, 32);
    sp.omega = fe_to_mont<Fr>(root);
    for (uint32_t i = k; i < (uint32_t)FR_S; ++i) sp.omega = fe_sqr<Fr>(sp.omega);
    fe sn = sp.s;
    for (uint32_t i = 0; i < k; ++i) sn = fe_sqr<Fr>(sn);                       // s^(2^k)
    sp.mult = fe_mul<Fr>(fe_sub<Fr>(sn, fe_one<Fr>()), fe_inv<Fr>(fr_from_small((uint64_t)n)));
    if (fe_is_zero(fe_sub<Fr>(sn, fe_one<Fr>()))) return failf(H2V_EINVAL, "srs_setup: s is a 2^k-th root of unity");
    DevBuf O;
    if ((rc = O.ensure(n * sizeof(affine)))) return rc;
    uint64_t *dst[2] = {g_out, g_lagrange_out};
    for (int b = 0; b < 2; ++b) {
        if (!dst[b]) continue;
        srs_setup_kernel<<<(unsigned)((n + 127) / 128), 128>>>(sp, b, O.as<affine>());
        H2V_LAUNCHED();
        H2V_CU(cudaDeviceSynchronize());
        H2V_CU(cudaMemcpy(dst[b], O.p, n * sizeof(affine), cudaMemcpyDeviceToHost));
    }
    O.release();
    return H2V_OK;
}
int h2v_synthetic_bases(uint64_t a, uint64_t b, size_t n, uint64_t *out_affine) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!out_affine || n == 0) return failf(H2V_EINVAL, "synthetic_bases: bad argument");
    if (a >> 62 || b >> 62 || n >> 32) return failf(H2V_EINVAL, "synthetic_bases: a, b < 2^62 and n < 2^32 required");
    DevBuf O;
    if ((rc = O.ensure(n * 64))) return rc;
    synthetic_bases_kernel<<<(unsigned)((n + 127) / 128), 128>>>(O.as<affine>(), a, b, n);
    H2V_LAUNCHED();
    H2V_CU(cudaDeviceSynchronize());
    H2V_CU(cudaMemcpy(out_affine, O.p, n * 64, cudaMemcpyDeviceToHost));
    O.release();
    return H2V_OK;
}
// which: 0 Fq mul, one dependent chain per thread; 1 Fq mul, two chains; 2 XYZZ mixed add chain.
// Returns operations per second over the whole GPU.
int h2v_selftest_op_rate(int which, double *out) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!out || which < 0 || which > 2) return failf(H2V_EINVAL, "selftest_op_rate: bad argument");
    DevBuf O;
    if ((rc = O.ensure(256))) return rc;
    cudaDeviceProp prop;
    H2V_CU(cudaGetDeviceProperties(&prop, g_devs[0]));
    cudaEvent_t e0, e1;
    H2V_CU(cudaEventCreate(&e0));
    H2V_CU(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 4; ++rep) {
        double ops;
        H2V_CU(cudaEventRecord(e0));
        if (which == 0) {
            unsigned blocks = prop.multiProcessorCount * 8, iters = 4096;
            mul_probe_kernel<1><<<blocks, 256>>>(O.as<fe>(), iters);
            ops = (double)blocks * 256 * iters;
        } else if (which == 1) {
            unsigned blocks = prop.multiProcessorCount * 8, iters = 2048;
            mul_probe_kernel<2><<<blocks, 256>>>(O.as<fe>(), iters);
            ops = (double)blocks * 256 * iters * 2;
        } else {
            unsigned blocks = prop.multiProcessorCount * 16, iters = 512;
            madd_probe_kernel<<<blocks, 128>>>(O.as<xyzz>(), iters);
            ops = (double)blocks * 128 * iters;
        }
        H2V_LAUNCHED();
        H2V_CU(cudaEventRecord(e1));
        H2V_CU(cudaEventSynchronize(e1));
        float ms = 0;
        H2V_CU(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    O.release();
    *out = best;
    return H2V_OK;
}
int h2v_selftest_imad_peak(double *out);
// which 0: the loop-variant stream of round 1 (one xorshift update per 8 multiply-adds); 1: the pure chain probe
int h2v_selftest_imad_probe(int which, double *out) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!out || which < 0 || which > 1) return failf(H2V_EINVAL, "selftest_imad_probe: bad argument");
    if (which == 0) return h2v_selftest_imad_peak(out);
    DevBuf O;
    if ((rc = O.ensure(64))) return rc;
    cudaDeviceProp prop;
    H2V_CU(cudaGetDeviceProperties(&prop, g_devs[0]));
    cudaEvent_t e0, e1;
    H2V_CU(cudaEventCreate(&e0));
    H2V_CU(cudaEventCreate(&e1));
    double best = 0;
    for (int occ = 2; occ <= 8; occ *= 2) {          // resident CTAs per SM: the rate must not depend on it once the pipe is full
        const unsigned blocks = prop.multiProcessorCount * occ, threads = 256, iters = 1 << 12;
        for (int rep = 0; rep < 3; ++rep) {
            H2V_CU(cudaEventRecord(e0));
            imad_chain_probe_kernel<<<blocks, threads>>>(O.as<uint32_t>(), iters, 777u + rep);
            H2V_LAUNCHED();
            H2V_CU(cudaEventRecord(e1));
            H2V_CU(cudaEventSynchronize(e1));
            float ms = 0;
            H2V_CU(cudaEventElapsedTime(&ms, e0, e1));
            const double rate = (double)blocks * threads * iters * 64.0 / (ms * 1e-3);      // 16 rows x 4 per iteration
            if (rep > 0 && rate > best) best = rate;
        }
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    O.release();
    *out = best;
    return H2V_OK;
}
int h2v_selftest_imad_peak(double *out) {
    int rc = use_device(g_devs[0]);
    if (rc) return rc;
    if (!out) return failf(H2V_EINVAL, "selftest_imad_peak: NULL");
    DevBuf O;
    if ((rc = O.ensure(64))) return rc;
    cudaDeviceProp prop;
    H2V_CU(cudaGetDeviceProperties(&prop, g_devs[0]));
    const unsigned blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
    cudaEvent_t e0, e1;
    H2V_CU(cudaEventCreate(&e0));
    H2V_CU(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        H2V_CU(cudaEventRecord(e0));
        imad_probe_kernel<<<blocks, threads>>>(O.as<uint64_t>(), iters, 12345u + rep);
        H2V_LAUNCHED();
        H2V_CU(cudaEventRecord(e1));
        H2V_CU(cudaEventSynchronize(e1));
        float ms = 0;
        H2V_CU(cudaEventElapsedTime(&ms, e0, e1));
        double rate = (double)blocks * threads * iters * 8.0 / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    O.release();
    *out = best;
    return H2V_OK;
}
}

namespace {
// a replica of `src` on device `dev`: the window tables cross NVLink / PCIe once (peer copy)
int rep_srs_clone(int dev, const SrsRep *src, SrsRep **out) {
    int rc = use_device(dev);
    if (rc) return rc;
    SrsRep *s = new SrsRep();
    s->dev = dev;
    s->k = src->k;
    s->n = src->n;
    s->cfg[0] = src->cfg[0];
    s->cfg[1] = src->cfg[1];
    s->have_small = src->have_small;
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete s;
        return failf(H2V_ECUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    for (int b = 0; b < 2; ++b) {
        if (!src->have[b]) continue;
        for (int v = 0; v < (s->have_small ? 2 : 1); ++v) {
            const size_t bytes = (size_t)s->cfg[v].W * s->n * sizeof(affine);
            rc = s->table[b][v].ensure(bytes);
            if (rc) { rep_srs_free(s); return rc; }
            e = cudaMemcpyPeerAsync(s->table[b][v].p, s->dev, src->table[b][v].p, src->dev, bytes, s->stream);
            if (e != cudaSuccess) { rep_srs_free(s); return failf(H2V_ECUDA, "SRS replica copy: %s", cudaGetErrorString(e)); }
        }
        s->have[b] = true;
    }
    e = cudaStreamSynchronize(s->stream);
    if (e != cudaSuccess) { rep_srs_free(s); return failf(H2V_ECUDA, "SRS replica copy: %s", cudaGetErrorString(e)); }
    *out = s;
    return H2V_OK;
}
// run fn(reps[i], i) for every replica, each on a host thread of its own (reps[0] on the calling thread, whose current
// device is the same afterwards as before); first error wins
template <class Rep, class Fn> int fan_out(const std::vector<Rep *> &reps, Fn fn) {
    int home = 0;
    cudaGetDevice(&home);
    const size_t n_slots = reps.size();
    std::vector<int> rcs(n_slots, H2V_OK);
    std::vector<std::string> errs(n_slots);
    std::vector<std::thread> th;
    for (size_t i = 1; i < n_slots; ++i)
        th.emplace_back([&, i] {
            rcs[i] = fn(reps[i], i);
            if (rcs[i]) errs[i] = g_err;
        });
    rcs[0] = fn(reps[0], 0);
    if (rcs[0]) errs[0] = g_err;
    for (auto &t : th) t.join();
    cudaSetDevice(home);
    for (size_t i = 0; i < n_slots; ++i)
        if (rcs[i]) {
            g_err = errs[i];
            return rcs[i];
        }
    return H2V_OK;
}

// The replicas of a handle: make(dev, &rep) builds one per h2v_init device, in list order; on an error the ones built so
// far are freed, each on its own device.  Both leave the calling thread on the primary device.
template <class Rep> void free_replicas(std::vector<Rep *> &reps, void (*free_rep)(Rep *)) {
    for (Rep *r : reps) free_rep(r);
    reps.clear();
    cudaSetDevice(g_devs[0]);
}
template <class Rep, class Make> int make_replicas(std::vector<Rep *> &reps, void (*free_rep)(Rep *), Make make) {
    for (int dev : g_devs) {
        Rep *r = nullptr;
        const int rc = make(dev, &r);
        if (rc) {
            free_replicas(reps, free_rep);
            return rc;
        }
        reps.push_back(r);
    }
    cudaSetDevice(g_devs[0]);
    return H2V_OK;
}

// cnt columns of `bytes` each from device src_dev to device dst_dev, on st: one copy when both sides hold them
// contiguously, one per column otherwise
cudaError_t peer_copy(void *dst, size_t dst_stride, int dst_dev, const void *src, size_t src_stride, int src_dev, size_t bytes, size_t cnt,
                      cudaStream_t st) {
    if (dst_stride == bytes && src_stride == bytes) return cudaMemcpyPeerAsync(dst, dst_dev, src, src_dev, cnt * bytes, st);
    cudaError_t e = cudaSuccess;
    for (size_t c = 0; c < cnt && e == cudaSuccess; ++c)
        e = cudaMemcpyPeerAsync((char *)dst + c * dst_stride, dst_dev, (const char *)src + c * src_stride, src_dev, bytes, st);
    return e;
}

bool peer_split_allowed() {
    static const bool no_split = getenv("H2V_NO_PEER_SPLIT") != nullptr;      // keep resident batches on their owner (tuning)
    return !no_split;
}
// Several devices, one resident batch on `owner`'s device (a phase of create_proof): the columns are independent, so the
// batch is cut into one contiguous block per replica.  The owner runs its block in place; every other replica pulls its
// block over NVLink, runs it and pushes the results back into the owner's output.  No collective; results in column
// order.  A column is in_bytes of input, in_stride bytes apart, and out_bytes of result, out_stride bytes apart.
// run(rep, in, in_stride, out, out_stride, count) runs `count` columns on `rep` (strides in bytes); a pulled block is
// packed, and its results are out_stride apart.
template <class Rep, class Run>
int split_blocks(const std::vector<Rep *> &reps, Rep *owner, const char *what, const void *in, size_t in_bytes, size_t in_stride, void *out,
                 size_t out_bytes, size_t out_stride, size_t n_cols, Run run) {
    const size_t per = (n_cols + reps.size() - 1) / reps.size();
    const char *src = (const char *)in;
    char *dst = (char *)out;
    return fan_out(reps, [&](Rep *rep, size_t d) -> int {
        const size_t c0 = std::min(n_cols, d * per), cnt = std::min(n_cols, c0 + per) - c0;
        if (!cnt) return H2V_OK;
        if (rep == owner) return run(rep, src + c0 * in_stride, in_stride, dst + c0 * out_stride, out_stride, cnt);
        H2V_TRY(use_device(rep->dev));
        std::lock_guard<std::mutex> plk(rep->peer_mu);
        {
            std::lock_guard<std::mutex> lk(rep->mu);
            H2V_TRY(rep->peer_in.ensure(cnt * in_bytes));
            H2V_TRY(rep->peer_out.ensure(cnt * out_stride));
            cudaError_t e = peer_copy(rep->peer_in.p, in_bytes, rep->dev, src + c0 * in_stride, in_stride, owner->dev, in_bytes, cnt, rep->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(rep->stream);
            if (e != cudaSuccess) return failf(H2V_ECUDA, "%s: peer copy %d -> %d: %s", what, owner->dev, rep->dev, cudaGetErrorString(e));
        }
        H2V_TRY(run(rep, rep->peer_in.p, in_bytes, rep->peer_out.p, out_stride, cnt));
        // (cudaMemcpyPeer returns before the copy has landed and does not order against non-blocking streams: copy on the
        // replica's stream and wait for it)
        cudaError_t e = peer_copy(dst + c0 * out_stride, out_stride, owner->dev, rep->peer_out.p, out_stride, rep->dev, out_bytes, cnt, rep->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(rep->stream);
        if (e != cudaSuccess) return failf(H2V_ECUDA, "%s: peer copy of the results: %s", what, cudaGetErrorString(e));
        return H2V_OK;
    });
}

// Host columns over several devices: column j goes to replica j mod G (each device has its own PCIe link and replica, no
// collective).  run(rep, in, out, count) gets the replica's input and output columns in column order.
template <class Rep, class In, class Out, class Run> int deal_columns(const std::vector<Rep *> &reps, const In *in, const Out *out, size_t n, Run run) {
    const size_t G = reps.size();
    std::vector<std::vector<In>> si(G);
    std::vector<std::vector<Out>> so(G);
    for (size_t j = 0; j < n; ++j) {
        si[j % G].push_back(in[j]);
        so[j % G].push_back(out[j]);
    }
    return fan_out(reps, [&](Rep *rep, size_t d) { return run(rep, si[d].data(), so[d].data(), si[d].size()); });
}
}  // namespace

extern "C" {

int h2v_dev_alloc_on(int device, size_t bytes, void **d_out) {
    bool known = false;
    for (int d : g_devs) known = known || d == device;
    if (!known) return failf(H2V_EINVAL, "dev_alloc_on: device %d is not in the h2v_init list", device);
    if (!d_out || !bytes) return failf(H2V_EINVAL, "dev_alloc: bad argument");
    H2V_TRY(use_device(device));
    cudaError_t e = cudaMalloc(d_out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return failf(H2V_ENOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
    }
    return H2V_OK;
}

// ---------------------------------------------------------------- SRS
int h2v_srs_load(uint32_t k, const uint64_t *g, const uint64_t *g_lagrange, h2v_srs_t *out) {
    if (!out) return failf(H2V_EINVAL, "h2v_srs_load: out is NULL");
    *out = nullptr;
    h2v_srs *h = new h2v_srs();
    const int rc = make_replicas(h->rep, rep_srs_free, [&](int dev, SrsRep **r) {
        return h->rep.empty() ? rep_srs_load(dev, k, g, g_lagrange, r) : rep_srs_clone(dev, h->rep[0], r);
    });
    if (rc) delete h;
    else *out = h;
    return rc;
}
void h2v_srs_free(h2v_srs_t h) {
    if (!h) return;
    free_replicas(h->rep, rep_srs_free);
    delete h;
}
int h2v_commit_batch_dev(h2v_srs_t h, int basis, const void *d_polys, size_t col_stride, size_t n_polys, size_t len, void *d_out_affine) {
    if (!h) return failf(H2V_EINVAL, "commit: NULL srs");
    SrsRep *r = srs_on(h, device_of(d_polys));
    if (!r) return failf(H2V_EINVAL, "commit: the columns live on device %d, which is not in the h2v_init list", device_of(d_polys));
    H2V_TRY(use_device(r->dev));
    const size_t G = h->rep.size();
    if (G == 1 || !peer_split_allowed() || n_polys < 8 * G || len == 0 || device_of(d_out_affine) != r->dev)
        return rep_commit_batch_dev(r, basis, d_polys, col_stride, n_polys, len, d_out_affine);
    // 32 B x len per column cross NVLink against ~10^3 x that in multiplier work; 64 B of commitment come back
    return split_blocks(h->rep, r, "commit", d_polys, len * sizeof(fe), col_stride * sizeof(fe), d_out_affine, sizeof(affine), sizeof(affine),
                        n_polys, [&](SrsRep *rep, const void *in, size_t in_stride, void *out, size_t, size_t cnt) {
                            return rep_commit_batch_dev(rep, basis, in, in_stride / sizeof(fe), cnt, len, out);
                        });
}
// Host columns that are committed AND left resident (the advice phase of create_proof): every device uploads a contiguous
// block of the columns over its own PCIe link in sub-batches (the next one crosses while the previous one is committed),
// overwrites the blinding rows, commits against its SRS replica and forwards the block to the destination buffer on the
// owning device over NVLink; commitments land in the host array in column order.
int h2v_commit_batch_resident(h2v_srs_t h, int basis, const uint64_t *const *polys, size_t n_polys, size_t len, const uint64_t *tails,
                              size_t row0, size_t n_rows, void *d_dst, size_t dst_stride, uint64_t *out_affine) {
    if (!h) return failf(H2V_EINVAL, "commit: NULL srs");
    if (n_polys == 0) return H2V_OK;
    if (!polys || !d_dst || !out_affine || (n_rows && !tails)) return failf(H2V_EINVAL, "commit_resident: NULL buffer");
    if (len == 0 || dst_stride < len || row0 + n_rows > len) return failf(H2V_EINVAL, "commit_resident: bad length / stride / row range");
    for (size_t c = 0; c < n_polys; ++c)
        if (!polys[c]) return failf(H2V_EINVAL, "commit_resident: polys[%zu] is NULL", c);
    SrsRep *r = srs_on(h, device_of(d_dst));
    if (!r) return failf(H2V_EINVAL, "commit_resident: the destination lives on device %d, which is not in the h2v_init list", device_of(d_dst));
    H2V_TRY(use_device(r->dev));
    const std::vector<SrsRep *> reps = h->rep.size() > 1 && n_polys >= 8 * h->rep.size() ? h->rep : std::vector<SrsRep *>{r};
    const size_t per = (n_polys + reps.size() - 1) / reps.size();
    fe *dst = (fe *)d_dst;
    return fan_out(reps, [&](SrsRep *rep, size_t d) -> int {
        const size_t c0 = std::min(n_polys, d * per), cnt = std::min(n_polys, c0 + per) - c0;
        if (!cnt) return H2V_OK;
        int rc2 = use_device(rep->dev);
        if (rc2) return rc2;
        const bool owner = rep == r;
        std::lock_guard<std::mutex> plk(rep->peer_mu);
        if (!owner && (rc2 = rep->peer_in.ensure(cnt * len * sizeof(fe)))) return rc2;
        if ((rc2 = rep->peer_out.ensure(cnt * sizeof(affine)))) return rc2;
        if (!rep->up_stream) H2V_CU(cudaStreamCreateWithFlags(&rep->up_stream, cudaStreamNonBlocking));
        fe *stage = owner ? dst + c0 * dst_stride : rep->peer_in.as<fe>();
        const size_t sstride = owner ? dst_stride : len;
        // few sub-batches: every commit call ends in a latency-bound reduction tail (~1 ms) that only size amortises
        const size_t sub = std::max<size_t>((cnt + 3) / 4, std::max<size_t>(1, ((size_t)64 << 20) / (len * sizeof(fe))));
        const size_t nsub = (cnt + sub - 1) / sub;
        std::vector<cudaEvent_t> ev(nsub, nullptr);
        cudaError_t e = cudaSuccess;
        for (size_t b = 0; b < nsub && e == cudaSuccess; ++b) {
            const size_t off = std::min(cnt, b * sub), m = std::min(cnt, off + sub) - off;
            if (m) e = stage_columns(true, stage + off * sstride, sstride, polys + c0 + off, m, len, rep->up_stream);
            if (m && n_rows && e == cudaSuccess)
                e = cudaMemcpy2DAsync(stage + off * sstride + row0, sstride * sizeof(fe), tails + (c0 + off) * n_rows * 4, n_rows * sizeof(fe),
                                      n_rows * sizeof(fe), m, cudaMemcpyHostToDevice, rep->up_stream);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventRecord(ev[b], rep->up_stream);
        }
        for (size_t b = 0; b < nsub && e == cudaSuccess && !rc2; ++b) {
            const size_t off = std::min(cnt, b * sub), m = std::min(cnt, off + sub) - off;
            if (!m) continue;
            e = cudaEventSynchronize(ev[b]);
            if (e != cudaSuccess) break;
            rc2 = rep_commit_batch_dev(rep, basis, stage + off * sstride, sstride, m, len, rep->peer_out.as<affine>() + off);
            if (rc2 || owner) continue;
            e = peer_copy(dst + (c0 + off) * dst_stride, dst_stride * sizeof(fe), r->dev, stage + off * len, len * sizeof(fe), rep->dev,
                          len * sizeof(fe), m, rep->up_stream);
        }
        if (e == cudaSuccess && !rc2)
            e = cudaMemcpyAsync(out_affine + 8 * c0, rep->peer_out.p, cnt * sizeof(affine), cudaMemcpyDeviceToHost, rep->up_stream);
        cudaError_t e2 = cudaStreamSynchronize(rep->up_stream);
        for (cudaEvent_t x : ev)
            if (x) cudaEventDestroy(x);
        if (rc2) return rc2;
        if (e != cudaSuccess || e2 != cudaSuccess)
            return failf(H2V_ECUDA, "commit_resident: %s", cudaGetErrorString(e != cudaSuccess ? e : e2));
        return H2V_OK;
    });
}
// Host columns: with several devices column j goes to device j mod G; the commitments come back in column order.
int h2v_commit_batch(h2v_srs_t h, int basis, const uint64_t *const *polys, size_t n_polys, size_t len, uint64_t *out_affine) {
    if (!h) return failf(H2V_EINVAL, "commit: NULL srs");
    H2V_TRY(use_device(h->rep[0]->dev));
    const size_t G = h->rep.size();
    if (G == 1 || n_polys < 2 * G || !polys || !out_affine) return rep_commit_batch(h->rep[0], basis, polys, n_polys, len, out_affine);
    std::vector<uint64_t *> outs(n_polys);
    for (size_t j = 0; j < n_polys; ++j) outs[j] = out_affine + 8 * j;
    return deal_columns(h->rep, polys, outs.data(), n_polys, [&](SrsRep *rep, const uint64_t *const *in, uint64_t *const *out, size_t cnt) {
        std::vector<uint64_t> res(8 * cnt);
        const int rc = rep_commit_batch(rep, basis, in, cnt, len, res.data());
        for (size_t i = 0; i < cnt && !rc; ++i) memcpy(out[i], &res[8 * i], 64);
        return rc;
    });
}
int h2v_commit(h2v_srs_t h, int basis, const uint64_t *poly, size_t len, uint64_t out_affine[8]) {
    if (!h) return failf(H2V_EINVAL, "commit: NULL srs");
    return rep_commit_batch(h->rep[0], basis, &poly, 1, len, out_affine);
}

// ---------------------------------------------------------------- EvaluationDomain
int h2v_domain_new(uint32_t j, uint32_t k, h2v_domain_t *out) {
    if (!out) return failf(H2V_EINVAL, "domain_new: out is NULL");
    *out = nullptr;
    h2v_domain *h = new h2v_domain();
    const int rc = make_replicas(h->rep, rep_domain_free, [&](int dev, DomRep **r) { return rep_domain_new(dev, j, k, r); });
    if (rc) delete h;
    else *out = h;
    return rc;
}
void h2v_domain_free(h2v_domain_t h) {
    if (!h) return;
    free_replicas(h->rep, rep_domain_free);
    delete h;
}
int h2v_domain_transform_dev(h2v_domain_t h, int op, const void *d_in, size_t in_stride, void *d_out, size_t out_stride, size_t n_cols) {
    DomRep *r = dom_rep(h, d_in);
    if (!r) return H2V_EINVAL;
    H2V_TRY(use_device(r->dev));
    const size_t G = h->rep.size();
    // worth splitting when every device gets about 2^21 points of transform: 8 columns of a 2^18-point extended domain
    // (k = 16), a single column from 2^21 points up (k = 20: one coset transform is 0.8 ms, its NVLink round trip 0.2 ms)
    const bool known_op = op >= 0 && op <= H2V_OP_DIVIDE_BY_VANISHING;
    const size_t work_len = (size_t)1 << (op >= H2V_OP_COEFF_TO_EXTENDED ? r->ek : r->k);
    const size_t min_per_dev = std::min<size_t>(8, std::max<size_t>(1, ((size_t)1 << 21) / (known_op ? work_len : 1)));
    const size_t nin = op_in_len(r, op), nout = op_out_len(r, op);
    if (G == 1 || !peer_split_allowed() || n_cols < min_per_dev * G || !known_op || !d_out || device_of(d_out) != r->dev || in_stride < nin ||
        out_stride < work_len)
        return rep_domain_transform_dev(r, op, d_in, in_stride, d_out, out_stride, n_cols);
    // 32 B per input element in, 32 B per output element out: worth it for the extended transforms, whose 4n-point
    // butterflies dominate
    return split_blocks(h->rep, r, "transform", d_in, nin * sizeof(fe), in_stride * sizeof(fe), d_out, nout * sizeof(fe), out_stride * sizeof(fe),
                        n_cols, [&](DomRep *rep, const void *in, size_t in_st, void *out, size_t out_st, size_t cnt) {
                            return rep_domain_transform_dev(rep, op, in, in_st / sizeof(fe), out, out_st / sizeof(fe), cnt);
                        });
}
int h2v_domain_transform_batch(h2v_domain_t h, int op, const uint64_t *const *in, uint64_t *const *out, size_t n_cols) {
    if (!h) return failf(H2V_EINVAL, "transform: NULL domain");
    H2V_TRY(use_device(h->rep[0]->dev));
    const size_t G = h->rep.size();
    if (G == 1 || n_cols < 2 * G || !in || !out) return rep_domain_transform_batch(h->rep[0], op, in, out, n_cols);
    return deal_columns(h->rep, in, out, n_cols, [&](DomRep *rep, const uint64_t *const *i, uint64_t *const *o, size_t cnt) {
        return rep_domain_transform_batch(rep, op, i, o, cnt);
    });
}

}  // extern "C"
