"""The step before the hot path (SURVEY.md 8(f) row 4): the reference's chips on the host and the column layout.

Modelled on the reference's own tests (/root/reference/tests/distances_test.rs, vectordb_test.rs: chip results against
f64 computations with `assert_float_relative_eq!`, epsilon 1e-6) plus what its `mock` command checks
(/root/reference/src/scaffold/mod.rs:263-266, MockProver): every gate, lookup and copy constraint of the laid-out circuit.
The checkers live in oracle/mock.py; the cell counts of the product's builder are compared with an independently written
count.  GPU: the laid-out circuits go through h2v_create_proof and the restated verifier accepts the proofs."""
import json
import math
import os

import numpy as np
import pytest

from oracle import mock as M
from oracle import oracle as O
from oracle import plonk as PL
from oracle import pyref as P
from oracle import transcript as T

EPS = 1e-6      # assert_float_eq's default for assert_float_relative_eq!


def rel_eq(a, b, eps=EPS):
    return abs(a - b) <= eps * max(abs(a), abs(b)) or abs(a - b) < 1e-12


@pytest.fixture(scope="module")
def Z():
    from halo2_vectordb_b200 import circuit as z

    return z


def _chips(Z, lookup_bits=13):
    b = Z.GateThreadBuilder.mock(lookup_bits)
    fp = Z.FixedPointChip.default(b)
    return b, b.main(0), fp


def _ints(cols):
    return [O.fr_to_ints(np.ascontiguousarray(c)) for c in cols]


def _trace_gates_hold(b):
    adv, sel, lk = b.trace()
    vals = O.limbs_to_ints(adv)
    assert len(sel) == len(vals)
    bad = [i for i in np.nonzero(sel)[0] if (vals[i] + vals[i + 1] * vals[i + 2] - vals[i + 3]) % P.R]
    table = 1 << b.lookup_bits
    out_of_table = [int(i) for i in lk if vals[i] >= table]
    return bad, out_of_table


# ----------------------------------------------------------------------------------------------- fixed point
def test_quantization_round_trip(Z):
    b, ctx, fp = _chips(Z)
    xs = [0.0, 1.0, -1.0, 0.5, -0.5, 3.141592653589793, -2.718281828, 123456.789, -98765.4321, 1e-9, -1e-9]
    q = fp.quantize_vector(xs)
    ints = O.fr_to_ints(q)
    for x, v in zip(xs, ints):
        want = round(abs(x) * 2 ** 48)
        assert v == (want if x >= 0 else (P.R - want) % P.R)      # fixed_point.rs:104-119
    back = fp._deq(q)
    for x, y, v in zip(xs, back, ints):
        # dequantization of a negative is off by two units in the last place (fixed_point.rs:123-125): bn254_max - x - 1
        assert abs(x - y) <= 3 / 2 ** 48 + abs(x) * 2 ** -52, (x, y)
    assert fp.dequantization(O.fr_from_ints([P.R - (1 << 48)])[0]) == -(1.0 - 2 / 2 ** 48)


@pytest.mark.parametrize("name,fn", [
    ("qadd", lambda a, b: a + b), ("qsub", lambda a, b: a - b), ("qmul", lambda a, b: a * b), ("qdiv", lambda a, b: a / b),
    ("qmax", max), ("qmin", min), ("qpow", lambda a, b: abs(a) ** b)])
def test_fixed_point_binary_ops(Z, name, fn):
    b, ctx, fp = _chips(Z)
    rng = np.random.default_rng(hash(name) % 1000)
    for _ in range(4):
        x, y = (float(v) for v in rng.uniform(-4, 4, 2))
        if name == "qpow":
            x = abs(x) + 0.1
        a, c = ctx.assign_witnesses(fp.quantize_vector([x, y]))
        got = fp.dequantization(getattr(fp, name)(ctx, a, c).value())
        assert rel_eq(got, fn(x, y), 2e-6 if name == "qpow" else EPS), (name, x, y, got)
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


@pytest.mark.parametrize("name,fn,lo,hi", [
    ("qabs", abs, -5, 5), ("neg", lambda a: -a, -5, 5), ("qexp2", lambda a: 2 ** a, -6, 6), ("qlog2", math.log2, 0.01, 100),
    ("qexp", math.exp, -4, 4), ("qlog", math.log, 0.01, 100), ("qsqrt", math.sqrt, 0.01, 100), ("qsin", math.sin, -6, 6),
    ("qcos", math.cos, -6, 6), ("qtan", math.tan, -1.2, 1.2), ("qsinh", math.sinh, -3, 3), ("qcosh", math.cosh, -3, 3),
    ("qtanh", math.tanh, -3, 3)])
def test_fixed_point_unary_ops(Z, name, fn, lo, hi):
    b, ctx, fp = _chips(Z)
    rng = np.random.default_rng(len(name))
    for _ in range(3):
        x = float(rng.uniform(lo, hi))
        a = ctx.load_witness(fp.quantization(x))
        got = fp.dequantization(getattr(fp, name)(ctx, a).value())
        assert abs(got - fn(x)) <= 5e-6 * max(1.0, abs(fn(x))), (name, x, got, fn(x))
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


def test_sign_predicates(Z):
    b, ctx, fp = _chips(Z)
    one = O.fr_to_ints(fp.quantization(1.0))[0]
    for x in (2.5, -2.5, 0.0):
        a = ctx.load_witness(fp.quantization(x))
        assert O.fr_to_ints(fp.is_neg(ctx, a).value())[0] == (1 if x < 0 else 0)
        assert O.fr_to_ints(fp.sign(ctx, a).value())[0] == (P.R - 1 if x < 0 else 1)
        assert fp.dequantization(fp.clip(ctx, a).value()) == pytest.approx(x, abs=1e-12)
    t, f = ctx.load_witness(O.fr_from_ints([1])[0]), ctx.load_witness(O.fr_from_ints([0])[0])
    assert [O.fr_to_ints(fp.bit_xor(ctx, p, q).value())[0] for p, q in ((t, t), (t, f), (f, t), (f, f))] == [0, 1, 1, 0]
    a = ctx.load_witness(fp.quantization(1.5))
    assert fp.dequantization(fp.cond_neg(ctx, a, t).value()) == pytest.approx(-1.5)
    assert fp.dequantization(fp.cond_neg(ctx, a, f).value()) == pytest.approx(1.5)
    xs = ctx.assign_witnesses(fp.quantize_vector([0.5, -1.25, 2.0]))
    assert fp.dequantization(fp.qsum(ctx, xs).value()) == pytest.approx(1.25)
    ys = ctx.assign_witnesses(fp.quantize_vector([2.0, 4.0, -1.0]))
    assert fp.dequantization(fp.inner_product(ctx, xs, ys).value()) == pytest.approx(0.5 * 2 - 1.25 * 4 - 2.0, abs=1e-9)
    coef = ctx.assign_witnesses(fp.quantize_vector([2.0, -3.0, 0.5]))      # 2 x^2 - 3 x + 0.5, highest degree first
    assert fp.dequantization(fp.polynomial(ctx, xs[2], coef).value()) == pytest.approx(2 * 4 - 6 + 0.5, abs=1e-9)
    assert one == 1 << 48
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


def test_chip_panics_surface_as_errors(Z):
    b, ctx, fp = _chips(Z)
    a, z = ctx.assign_witnesses(fp.quantize_vector([1.0, 0.0]))
    with pytest.raises(ValueError, match="divide by zero"):
        fp.qdiv(ctx, a, z)
    with pytest.raises(ValueError):
        Z.DistanceChip.default(fp).euclidean_distance(ctx, [a], [a, z])      # assert_eq!(a.len(), b.len())
    with pytest.raises(ValueError, match="K < vectors.len"):
        Z.VectorDBChip.default(fp).kmeans(ctx, [[a], [z]], Z.DISTANCE_EUCLIDEAN, 2, 1)
    with pytest.raises(ValueError, match="precision"):
        Z.GateThreadBuilder(12, precision_bits=20)
    with pytest.raises(ValueError):
        b.call(Z.FP_QADD, [a])
    with pytest.raises(ValueError):
        b.call(Z.FP_QADD, [a, Z.AssignedValue(b, 10 ** 9)])


# ----------------------------------------------------------------------------------------------- distances (tests/distances_test.rs)
DIM = 10


def _native_distance(name, a, b):
    if name == "euclidean":
        return math.sqrt(sum((x - y) ** 2 for x, y in zip(a, b)))
    if name == "manhattan":
        return sum(abs(x - y) for x, y in zip(a, b))
    if name == "cosine":
        ab, aa, bb = sum(x * y for x, y in zip(a, b)), sum(x * x for x in a), sum(y * y for y in b)
        return 1.0 - ab / (math.sqrt(aa) * math.sqrt(bb))
    return 1.0 - sum(1.0 if x == y else 0.0 for x, y in zip(a, b)) / len(a)


@pytest.mark.parametrize("name", ["euclidean", "manhattan", "cosine", "hamming"])
def test_distance_matches_native(Z, name):
    rng = np.random.default_rng(7)
    for trial in range(3):
        a, c = [float(v) for v in rng.random(DIM)], [float(v) for v in rng.random(DIM)]
        if name == "hamming":
            c[2], c[5] = a[2], a[5]
        b, ctx, fp = _chips(Z)
        dist = Z.DistanceChip.default(fp)
        qa, qb = ctx.assign_witnesses(fp.quantize_vector(a)), ctx.assign_witnesses(fp.quantize_vector(c))
        got = fp.dequantization(getattr(dist, name + "_distance")(ctx, qa, qb).value())
        assert rel_eq(got, _native_distance(name, a, c)), (name, got)
        bad, oot = _trace_gates_hold(b)
        assert not bad and not oot


# ----------------------------------------------------------------------------------------------- vectordb (tests/vectordb_test.rs)
def _native_kmeans(vectors, K, I, dist):
    n = len(vectors[0])
    cent = [list(v) for v in vectors[:K]]
    ids = [0] * len(vectors)
    for _ in range(I):
        sizes = [0] * K
        for i, v in enumerate(vectors):
            d = [dist(v, c) for c in cent]
            ids[i] = d.index(min(d))
            sizes[ids[i]] += 1
        for c in range(K):
            mean = [0.0] * n
            for i, v in enumerate(vectors):
                if ids[i] == c:
                    for j in range(n):
                        mean[j] += v[j]
            cent[c] = [m / sizes[c] for m in mean]
    return cent, ids


def test_kmeans_small(Z):
    K, I, dim = 2, 4, 5
    rng = np.random.default_rng(11)
    vectors = [[float(x) for x in rng.random(dim)] for _ in range(30)]
    cent_n, ids_n = _native_kmeans(vectors, K, I, lambda a, b: _native_distance("euclidean", a, b))
    b, ctx, fp = _chips(Z)
    vdb = Z.VectorDBChip.default(fp)
    q = [ctx.assign_witnesses(fp.quantize_vector(v)) for v in vectors]
    cent, ind = vdb.kmeans(ctx, q, Z.DISTANCE_EUCLIDEAN, K, I)
    cent_c = [fp.dequantize_vector(c) for c in cent]
    ids_c = [[x == 1.0 for x in fp.dequantize_vector(i)].index(True) for i in ind]
    assert ids_c == ids_n
    for a, c in zip(cent_n, cent_c):
        assert all(rel_eq(x, y) for x, y in zip(a, c))
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


def test_nearest_vector(Z):
    dim = 4
    rng = np.random.default_rng(12)
    query = [float(x) for x in rng.random(dim)]
    vectors = [[float(x) for x in rng.random(dim)] for _ in range(4)]
    d = [_native_distance("euclidean", v, query) for v in vectors]
    b, ctx, fp = _chips(Z)
    vdb = Z.VectorDBChip.default(fp)
    ind, res = vdb.nearest_vector(ctx, ctx.assign_witnesses(fp.quantize_vector(query)),
                                  [ctx.assign_witnesses(fp.quantize_vector(v)) for v in vectors], Z.DISTANCE_EUCLIDEAN)
    assert [O.fr_to_ints(i.value())[0] for i in ind] == [1 if i == d.index(min(d)) else 0 for i in range(4)]
    assert all(rel_eq(x, y) for x, y in zip(fp.dequantize_vector(res), vectors[d.index(min(d))]))
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


def test_poseidon_chip_matches_native_sponge(Z):
    """the in-circuit sponge (optimised constants, sparse partial rounds, laid out as gates) against the oracle's plain
    Poseidon sponge, which the published `poseidonperm_x5_254_3` vector pins (tests/test_external_vectors.py)"""
    b, ctx, fp = _chips(Z, 12)
    pos = Z.PoseidonChip(ctx, 8, 57)
    for m in (1, 2, 3, 4, 5):
        vals = [(0x1234567 * (i + 1) ** 3 + m) % P.R for i in range(m)]
        cells = ctx.assign_witnesses(O.fr_from_ints(vals))
        pos.clear()
        pos.update(cells)
        got = O.fr_to_ints(pos.squeeze(ctx).value())[0]
        sp = T.PoseidonSponge(t=3, rate=2, r_f=8, r_p=57)
        sp.update(vals)
        assert got == sp.squeeze(), m
    bad, oot = _trace_gates_hold(b)
    assert not bad and not oot


def test_merkle_commitment(Z):
    b, ctx, fp = _chips(Z, 12)
    vdb = Z.VectorDBChip.default(fp)
    pos = Z.PoseidonChip(ctx, 8, 57)
    vecs = [[0.5 * i + j for j in range(3)] for i in range(5)]
    q = [ctx.assign_witnesses(fp.quantize_vector(v)) for v in vecs]
    root = O.fr_to_ints(vdb.merkle_commitment(ctx, pos, q).value())[0]

    def h(xs):
        sp = T.PoseidonSponge(t=3, rate=2, r_f=8, r_p=57)
        sp.update(xs)
        return sp.squeeze()

    leaves = [h(O.fr_to_ints(fp.quantize_vector(v))) for v in vecs] + [0] * 3      # padded to 8 leaves with zeros
    while len(leaves) > 1:
        leaves = [h(leaves[i:i + 2]) for i in range(0, len(leaves), 2)]
    assert root == leaves[0]


# ----------------------------------------------------------------------------------------------- examples, cell counts, layout
@pytest.mark.parametrize("name", ["distances", "query", "kmeans"])
def test_example_cell_counts_match_independent_count(Z, name):
    k, lb = Z.EXAMPLE_PARAMS[name]
    inp = Z.example_input(name)
    b = Z.GateThreadBuilder(lb)
    pub = []
    out = Z.EXAMPLES[name](b.main(0), inp, pub)
    b.make_public(pub)
    st = b.stats()
    assert (st["advice_cells"], st["lookup_cells"]) == M.example_cell_counts(name, inp, lb)
    cfg = b.config(k)
    max_rows = (1 << k) - 9
    assert cfg["num_advice_per_phase"] == [-(-st["advice_cells"] // max_rows)]
    assert cfg["num_lookup_advice_per_phase"] == [-(-st["lookup_cells"] // max_rows)]
    assert cfg["num_fixed"] == 1
    if name == "distances":
        want = {n: _native_distance(n, inp["a"], inp["b"]) for n in ("euclidean", "manhattan", "cosine", "hamming")}
        assert all(rel_eq(out[n], want[n]) for n in want), out
        assert st["instances"] == 4
    elif name == "query":
        assert all(rel_eq(x, y) for x, y in zip(out["result"], [0.111, 0.444, 1.777]))
    else:
        cent, ids = _native_kmeans(inp["vectors"], 4, 10, lambda a, c: _native_distance("cosine", a, c))
        assert all(rel_eq(x, y) for a, c in zip(cent, out["centroids"]) for x, y in zip(a, c))
        assert [[x == 1.0 for x in i].index(True) for i in out["indicators"]] == ids
        assert st["instances"] == 12


def test_example_inputs_are_the_reference_files(Z):
    """tests/golden/data holds the reference's example inputs (its data/{distances,query,kmeans}.in)"""
    ref = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data")
    for name in ("distances", "query", "kmeans"):
        with open(os.path.join(ref, name + ".in")) as f:
            assert json.load(f) == Z.example_input(name)


def _layout(Z, name, k=None, lookup_bits=None, inp=None, **kw):
    k0, lb0 = Z.EXAMPLE_PARAMS[name]
    return Z.create_circuit(Z.EXAMPLES[name], inp or Z.example_input(name), k or k0, lookup_bits or lb0, **kw)


def test_distances_layout_satisfies_mock_prover(Z):
    rc, _ = _layout(Z, "distances")
    assert (rc.num_advice, rc.num_lookup_advice, rc.num_fixed) == (9, 2, 1)
    assert len(rc.break_points) == rc.num_advice - 1 and all(bp >= (1 << 13) - 9 - 4 for bp in rc.break_points)
    fixed, sigma, advice, inst = _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances)
    assert M.mock_prover(rc.cs, fixed, sigma, advice, inst) == []
    assert len(inst[0]) == 4 and M.copy_classes(rc.cs, sigma) > 10000
    # a flipped witness cell, a wrong public input, a value outside the table: each is caught
    bad = [list(c) for c in advice]
    bad[0][7] = (bad[0][7] + 1) % P.R
    assert M.mock_prover(rc.cs, fixed, sigma, bad, inst)
    assert M.mock_prover(rc.cs, fixed, sigma, advice, [[(inst[0][0] + 1) % P.R] + inst[0][1:]])
    bad = [list(c) for c in advice]
    bad[rc.num_advice][3] = 1 << 12
    assert any("lookup" in f for f in M.mock_prover(rc.cs, fixed, sigma, bad, inst))


def test_query_layout(Z):
    """data/query.in repeats every database vector five times, so the minimum distance is attained five times and the
    indicator of nearest_vector has five ones; halo2-base's select_by_indicator fills its running cell assuming a one-hot
    indicator [UPSTREAM, recalled], which leaves exactly the gates of those repeated hits unsatisfied.  With the ties
    broken (a database of distinct vectors) the whole circuit is satisfied."""
    rc, _ = _layout(Z, "query")
    assert (rc.num_advice, rc.num_lookup_advice, rc.num_fixed) == (147, 19, 1)
    fails = M.mock_prover(rc.cs, _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances), max_failures=100)
    assert len(fails) == 12 and all(f.startswith("gate not satisfied") for f in fails)      # 3 coordinates x 4 repeated hits
    inp = Z.example_input("query")
    inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
    rc, out = _layout(Z, "query", inp=inp)
    assert M.mock_prover(rc.cs, _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances)) == []
    d = [_native_distance("cosine", v, inp["query"]) for v in inp["database"]]
    assert all(rel_eq(x, y) for x, y in zip(out["result"], inp["database"][d.index(min(d))]))


def test_layout_errors(Z):
    with pytest.raises(ValueError, match="LOOKUP_BITS"):
        _layout(Z, "distances", k=12, lookup_bits=12)
    b = Z.GateThreadBuilder(8)
    ctx = b.main(0)
    fp = Z.FixedPointChip.default(b)
    a, c = ctx.assign_witnesses(fp.quantize_vector([1.5, 2.5]))
    fp.qmul(ctx, a, c)
    b.make_public([a])
    with pytest.raises(ValueError):
        Z.RangeCircuit(b, 9, minimum_rows=600)      # minimum_rows >= 2^k
    rc = Z.RangeCircuit(b, 9)
    assert M.mock_prover(rc.cs, _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances)) == []
    # k = 9 leaves 503 rows per column: the trace breaks into several columns, each break repeats one cell
    assert rc.num_advice == -(-b.stats()["advice_cells"] // 503) and len(rc.break_points) == rc.num_advice - 1


def test_builder_symbols_exported(Z):
    import halo2_vectordb_b200 as h

    L = h.lib()
    assert [s for s in Z.BUILDER_SYMBOLS if not hasattr(L, s)] == []
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "h2v.h")).read()
    assert all(s + "(" in hdr for s in Z.BUILDER_SYMBOLS)


# ----------------------------------------------------------------------------------------------- GPU: real proofs of the real circuits
SEED = bytes(range(32))
SECRET = 0x1CE1CEBABE5EED0123456789ABCDEF0FEDCBA9876543210


def _prove_and_verify(h2v, rc, oracle_prover=False):
    k = rc.k
    s = O.fr_from_ints([SECRET])[0]
    g, gl = h2v.srs_setup(k, s)
    srs = h2v.ParamsKZG(k, g, gl)
    vk_repr = O.fr_from_ints([0x5eed])[0]
    pk = h2v.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, vk_repr)
    proof = pk.create_proof(rc.advice, rc.instances, SEED)
    # the verifying key's commitments come from the device too (commit parity has its own tests)
    vk = {"fixed": [O.g1_affine_to_ints(p) for p in srs.commit_batch(rc.fixed)],
          "sigma": [O.g1_affine_to_ints(p) for p in srs.commit_batch(rc.sigma)]}
    params = PL.Params(k, g, gl, SECRET)
    inst = _ints(rc.instances)
    ok = PL.verify_proof(params, rc.cs, vk, 0x5eed, inst, proof)
    bad_inst = [[(inst[0][0] + 1) % P.R] + inst[0][1:]]
    rejected = not PL.verify_proof(params, rc.cs, vk, 0x5eed, bad_inst, proof)
    same = None
    if oracle_prover:
        same = proof == PL.create_proof(params, rc.cs, _ints(rc.fixed), _ints(rc.sigma), 0x5eed, _ints(rc.advice), inst, SEED)
    pk.close()
    srs.close()
    return ok, rejected, same, proof


@pytest.mark.gpu
def test_gpu_proof_of_distances_example(h2v, Z):
    """BASELINE configs[0]: the distances example at k = 13, LOOKUP_BITS = 12 -- witness by the restated chips, proof by
    h2v_create_proof, bytes equal to the CPU restatement's, accepted by the restated verifier"""
    rc, out = _layout(Z, "distances")
    ok, rejected, same, proof = _prove_and_verify(h2v, rc, oracle_prover=True)
    assert ok and rejected and same
    # a proof of a tampered witness (one cell of the euclidean distance's trace) is rejected
    rc.advice[0][100, 0] ^= np.uint64(1)
    ok2, _, _, _ = _prove_and_verify(h2v, rc)
    assert not ok2


@pytest.mark.gpu
def test_gpu_proof_of_query_example(h2v, Z):
    """BASELINE configs[1] with the ties of data/query.in broken (see test_query_layout)"""
    inp = Z.example_input("query")
    inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
    rc, out = _layout(Z, "query", inp=inp)
    ok, rejected, _, proof = _prove_and_verify(h2v, rc)
    assert ok and rejected
    # the literal input: five-way ties leave select_by_indicator's gates unsatisfied, and the verifier says so
    rc2, _ = _layout(Z, "query")
    ok2, _, _, _ = _prove_and_verify(h2v, rc2)
    assert not ok2


@pytest.mark.gpu
def test_gpu_proof_of_kmeans_example(h2v, Z):
    """BASELINE configs[2]: kmeans (K = 4, I = 10, cosine) on data/kmeans.in at k = 16, LOOKUP_BITS = 15: 535 gate columns,
    72 lookup columns; the 20x target's circuit"""
    rc, out = _layout(Z, "kmeans")
    assert (rc.num_advice, rc.num_lookup_advice) == (535, 72)
    ok, rejected, _, proof = _prove_and_verify(h2v, rc)
    assert ok and rejected
