// internal.hpp -- helpers shared by the translation units of libh2v.so (not part of the C ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <vector>

#include "h2v.h"

namespace h2v {
int set_error(int code, const char *msg);     // h2v.cu: records the thread-local h2v_last_error() text
void count_launches(uint64_t n);              // h2v.cu: h2v_launch_count()
int current_device();

inline int failf(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    return set_error(code, buf);
}

// a device allocation that grows on demand and keeps its size between calls
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return H2V_OK;
        release();
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            return failf(H2V_ENOMEM, "cudaMalloc(%zu bytes): %s", bytes, cudaGetErrorString(e));
        }
        cap = bytes;
        return H2V_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// Entry points of the group prover (prover.cu), not part of the C ABI.
// Kate division of many device columns in one set of launches: job j divides a[0 .. n) by (X - b) into q[0 .. n - 1)
// (b: Montgomery limbs, as h2v_kate_division_dev takes it).  Synchronous.
struct KateJob {
    const void *a;
    void *q;
    size_t n;
    uint64_t b[4];
};
int kate_division_batch_dev(const KateJob *jobs, size_t n_jobs);
// evaluate_h's folds for n_proofs proofs, one launch per argument: proof p folds into h + p * h_stride with y, beta, gamma
// = scal[3p .. 3p + 2] (device); its gate table is n_gates selectors then n_gates advice columns at gate_tab + p * gate_pstride,
// its permutation table n_perm columns then n_perm sigma columns at perm_tab + p * perm_pstride, its products at
// z + p * z_pstride, its lookups 5 columns each (input, table, A', S', z) at lookup_tab + p * lookup_pstride.  Synchronous.
struct QuotientBatch {
    void *h;
    size_t h_stride;
    const void *scal;
    size_t n_proofs;
    size_t n_gates;
    const void *const *gate_tab;
    size_t gate_pstride;
    size_t n_perm, chunk;
    const void *const *perm_tab;
    size_t perm_pstride;
    const void *z;
    size_t z_stride, z_pstride;
    uint32_t blinding_factors;
    size_t n_lookups;
    const void *const *lookup_tab;
    size_t lookup_pstride;
    const void *l0, *l_last, *l_active;
};
int quotient_batch_dev(h2v_domain_t h, const QuotientBatch &b);

// The constraint-system checks of h2v_pk_load, in its order: degree, k, blinding factors, then "NULL column list" when
// have_column_lists is false, then every column index.  Errors name `who`.
int check_circuit(const h2v_circuit_t *cs, bool have_column_lists, const char *who);

// Launch helpers of h2v.cu over the lookup argument's kernels (lookup.cuh, msm.cuh), asynchronous on `st`.
struct fe;
// keys + s * n_pad <- the first u values of column d_srcs[s] (device pointer table), canonical and sorted ascending, padded
// with all-ones keys to n_pad (a power of two >= u), for s < slices
int sort_canonical_dev(cudaStream_t st, const fe *const *d_srcs, uint32_t slices, uint32_t u, uint32_t n_pad, fe *keys);
// offs = exclusive prefix sums of cnt[0 .. len), *total = their sum (device); tiles: ceil(len / 2048) words, scratch: len words
int scan_u32_dev(cudaStream_t st, const uint32_t *cnt, uint32_t len, uint32_t *offs, uint32_t *tiles, uint32_t *scratch, uint32_t *total);

// The mock prover's checks (mock.cu).  MockKey: what they need from the key alone (each permutation cell's image, the
// permutation's key-only flags, the sorted lookup tables), built once per key from its fixed and sigma columns on the
// device (Lagrange form, n rows each, contiguous).  The fixed columns must stay in place while the MockKey is used.
struct MockKey;
int mock_key_build(cudaStream_t st, const h2v_circuit_t *cs, const fe *fixed, const fe *sigma, MockKey **out);   // synchronous
void mock_key_free(MockKey *key);
size_t mock_witness_bytes(const MockKey &key);     // device bytes one witness of a check needs
size_t mock_max_batch(const MockKey &key);         // the most witnesses one mock_check takes
// B witnesses' host columns staged: witness w's advice columns uploaded to adv + w A n and its instance columns,
// zero-padded, to inst + w I n (prove_group's layout; adv and inst grow to fit).  ms[0] += the upload.  Synchronous.
int mock_stage(cudaStream_t st, const MockKey &key, size_t B, const uint64_t *const *const *advice, const uint64_t *const *const *instances,
               const uint32_t *const *instance_len, DevBuf &adv, DevBuf &inst, double ms[2]);
// B witnesses whose columns are resident in that layout checked: failures_out + w cap and n_failures[w] as
// h2v_mock_prover writes them.  ms[1] += the checks.  Synchronous.
int mock_check(cudaStream_t st, const MockKey &key, size_t B, const fe *adv, const fe *inst, h2v_mock_failure_t *failures_out, size_t cap,
               uint64_t *n_failures, double ms[2]);
void mock_set_last_ms(const double ms[2]);         // h2v_mock_last_ms
// the argument checks of h2v_mock_prover and h2v_pk_mock_prover; errors start with `who`
int mock_check_advice(const h2v_circuit_t *cs, const uint64_t *const *advice, const char *who);
int mock_check_instances(const h2v_circuit_t *cs, const uint64_t *const *instances, const uint32_t *instance_len, const char *who);
int mock_check_limits(const h2v_circuit_t *cs, const char *who);

// The group size for n_items items of item_bytes device bytes each when `held` bytes of device buffers can be reused:
// H2V_PROOF_GROUP if set, else as many as fit with 8 GB kept free; at most `cap` (prover.cu)
size_t group_size_free(size_t n_items, size_t item_bytes, size_t cap, size_t held);

// A witness program (circuit.cu builds it from a recording builder, witness.cu runs it).  Values are canonical.  An operand
// or gather reference is a slot (inputs first, then the computed cells in level order), WREF_POOL | i for constant i of the
// pool, or WREF_ZERO.
enum : uint32_t { WREF_POOL = 0x80000000u, WREF_ZERO = 0xffffffffu };
struct WitnessRule {
    uint32_t a, b, c;
    uint32_t op;      // zk::RuleKind | imm << 8
};
struct WitnessPlan {
    uint32_t k = 0, n_levels = 0;
    uint64_t n_inputs = 0, n_cells = 0, n_adv_cols = 0, n_instances = 0;
    std::vector<WitnessRule> rules;        // the computed cells, level by level
    std::vector<uint32_t> level_start;     // n_levels + 1 offsets into rules
    std::vector<uint64_t> cell_of;         // trace cell of each computed cell (error texts)
    std::vector<uint64_t> pool;            // 4 limbs per constant
    std::vector<uint32_t> map;             // 2^k rows of each advice column, then the instances
    std::vector<uint64_t> inputs;          // the recording's own inputs, Montgomery form
    std::vector<uint64_t> kind_counts;     // computed cells per zk::RuleKind
};
int witness_program_make(WitnessPlan &&plan, h2v_witness_program **out);      // witness.cu; takes the plan
bool fr_reduced(const uint64_t *x);      // 4 limbs below r
// A program run into a proving key's workspace (witness.cu).  The caller holds the program's mutex (after the key's).
std::mutex &witness_program_mutex(h2v_witness_program *p);
// The program on device dev, uploaded there in copies on st on first use (H2V_EINVAL naming `who` if it is resident on
// another device); the buffers of generated columns h2v_witness_generate grew are released and h2v_witness_last_ms starts
// from zero.  *held: the device bytes of the evaluation buffers the groups will reuse.
int witness_program_bind(h2v_witness_program *p, int dev, cudaStream_t st, const char *who, size_t *held);
size_t witness_eval_bytes(const h2v_witness_program *p);      // device bytes one witness's evaluation needs
// B witnesses (inputs: B x n_inputs x 4 limbs) evaluated and gathered on st: witness w's advice columns to adv + w A n,
// its instances to inst + w inst_stride, zero-padded to inst_stride rows, and to inst_host + w n_instances 4 unless
// inst_host is NULL; h2v_witness_last_ms accumulates.  A witness that panics: H2V_EINVAL with the panic text, *bad_w =
// the first such witness of the group (else B).  Synchronous.
int witness_generate_dev(h2v_witness_program *p, cudaStream_t st, size_t B, const uint64_t *inputs, fe *adv, fe *inst, size_t inst_stride,
                         uint64_t *inst_host, size_t *bad_w);
}  // namespace h2v

#define H2V_CU(x)                                                                                                  \
    do {                                                                                                           \
        cudaError_t e_ = (x);                                                                                      \
        if (e_ != cudaSuccess) return h2v::failf(H2V_ECUDA, "%s failed: %s", #x, cudaGetErrorString(e_));          \
    } while (0)
#define H2V_LAUNCHED()                                                                                             \
    do {                                                                                                           \
        h2v::count_launches(1);                                                                                    \
        cudaError_t e_ = cudaGetLastError();                                                                       \
        if (e_ != cudaSuccess)                                                                                     \
            return h2v::failf(H2V_ECUDA, "kernel launch failed (%s:%d): %s", __FILE__, __LINE__, cudaGetErrorString(e_)); \
    } while (0)
#define H2V_TRY(x)                  \
    do {                            \
        int rc_ = (x);              \
        if (rc_) return rc_;        \
    } while (0)
