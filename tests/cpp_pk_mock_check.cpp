// The C++ mirror of the mock prover on a loaded key (include/h2v.hpp): load h2v_host::ProvingKey from the circuit and
// columns in argv[1] (written by tests/test_pk_mock_prover.py::_write_case), check the witnesses there with
// ProvingKey::mock_prover and print "witness <w> <n_failures>" followed by one "<kind> <column> <row> <other_column>
// <other_row>" line per failure.  Without a device it prints "no device: ..." and exits 0.
#include <cstdio>
#include <cstring>
#include <fstream>
#include "h2v.hpp"
using namespace h2v_host;

namespace {
std::ifstream in;
uint32_t u32() {
    uint32_t v = 0;
    in.read(reinterpret_cast<char *>(&v), sizeof v);
    return v;
}
template <class T> std::vector<T> arr(size_t count) {
    std::vector<T> v(count);
    in.read(reinterpret_cast<char *>(v.data()), count * sizeof(T));
    return v;
}
std::vector<const Fr *> ptrs(const std::vector<Fr> &cols, size_t count, size_t n) {
    std::vector<const Fr *> p;
    for (size_t c = 0; c < count; ++c) p.push_back(cols.data() + c * n);
    return p;
}
}  // namespace

int main(int argc, char **argv) {
    if (h2v_device_count() <= 0) {
        try { init(0); } catch (const std::runtime_error &e) { std::printf("no device: %s\n", e.what()); return 0; }
        return 1;   // must have thrown
    }
    if (argc < 2) return 2;
    init(0);
    in.open(argv[1], std::ios::binary);
    h2v_circuit_t cs{};
    cs.k = u32(); cs.degree = u32(); cs.blinding_factors = u32();
    cs.n_advice = u32(); cs.n_fixed = u32(); cs.n_instance = u32();
    cs.n_gates = u32(); cs.n_lookups = u32(); cs.n_perm = u32(); cs.n_advice_queries = u32(); cs.n_fixed_queries = u32();
    const uint32_t B = u32(), cap = u32();
    const size_t n = size_t(1) << cs.k;
    auto gate_advice = arr<uint32_t>(cs.n_gates), gate_selector = arr<uint32_t>(cs.n_gates);
    auto lookup_input = arr<uint32_t>(cs.n_lookups), lookup_table = arr<uint32_t>(cs.n_lookups);
    auto perm_kind = arr<uint8_t>(cs.n_perm);
    auto perm_index = arr<uint32_t>(cs.n_perm);
    auto aq_col = arr<uint32_t>(cs.n_advice_queries);
    auto aq_rot = arr<int32_t>(cs.n_advice_queries);
    auto fq_col = arr<uint32_t>(cs.n_fixed_queries);
    auto fq_rot = arr<int32_t>(cs.n_fixed_queries);
    cs.gate_advice = gate_advice.data(); cs.gate_selector = gate_selector.data();
    cs.lookup_input = lookup_input.data(); cs.lookup_table = lookup_table.data();
    cs.perm_kind = perm_kind.data(); cs.perm_index = perm_index.data();
    cs.advice_query_col = aq_col.data(); cs.advice_query_rot = aq_rot.data();
    cs.fixed_query_col = fq_col.data(); cs.fixed_query_rot = fq_rot.data();
    auto g = arr<G1Affine>(n), gl = arr<G1Affine>(n);
    auto fixed = arr<Fr>(cs.n_fixed * n), sigma = arr<Fr>(cs.n_perm * n);
    const Fr vk = arr<Fr>(1)[0];
    std::vector<std::vector<Fr>> advice(B);
    std::vector<std::vector<const Fr *>> adv_ptrs(B);
    std::vector<std::vector<std::vector<Fr>>> instances(B);
    for (uint32_t w = 0; w < B; ++w) {
        advice[w] = arr<Fr>(cs.n_advice * n);
        adv_ptrs[w] = ptrs(advice[w], cs.n_advice, n);
        for (uint32_t c = 0; c < cs.n_instance; ++c) instances[w].push_back(arr<Fr>(u32()));
    }
    if (!in) { std::printf("short input\n"); return 3; }

    ParamsKZG params(cs.k, g, gl);
    ProvingKey pk(params, cs, ptrs(fixed, cs.n_fixed, n), ptrs(sigma, cs.n_perm, n), vk);
    const std::vector<MockProver> got = pk.mock_prover(adv_ptrs, instances, cap);
    for (uint32_t w = 0; w < B; ++w) {
        std::printf("witness %u %llu\n", w, (unsigned long long)got[w].n_failures);
        for (const auto &f : got[w].failures) std::printf("%u %u %u %u %u\n", f.kind, f.column, f.row, f.other_column, f.other_row);
    }
    bool threw = false;
    try { pk.mock_prover(adv_ptrs, {}, cap); } catch (const std::invalid_argument &) { threw = true; }
    if (!threw) return 4;
    return 0;
}
