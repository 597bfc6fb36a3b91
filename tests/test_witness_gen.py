"""Witness generation on the GPU (h2v_witness_generate): a recorded circuit replayed for many inputs must give, byte for
byte, the advice columns and instances a fresh host builder + RangeCircuit gives for each input.

The CPU tests check the recording and its premise: a recording builder's layout is the normal builder's, and the fixed
columns, sigma and break points of the example circuits do not depend on the input values.  The GPU tests compare the
generated columns with the host's for the examples, for one small program per chip operation over edge inputs, and
through create_proofs and the mock prover."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from oracle import pyref as P

R = P.R
PREC = 48


def _Z():
    from halo2_vectordb_b200 import circuit as Z

    return Z


def _layout_bytes(rc):
    return ([c.tobytes() for c in rc.advice], [c.tobytes() for c in rc.fixed], [c.tobytes() for c in rc.sigma],
            [i.tobytes() for i in rc.instances], rc.break_points)


def _example(Z, name, inp, record=False):
    k, bits = Z.EXAMPLE_PARAMS[name]
    return Z.create_circuit(Z.EXAMPLES[name], inp, k, bits, record=record)[0]


def _variants(Z, name):
    """the recording input, its negation, zeros, ties and random values, all of the recording's shape"""
    base = Z.example_input(name)
    rnd = random.Random(7)

    def mapv(f):
        return {key: ([[f(x) for x in v] for v in val] if isinstance(val[0], list) else [f(x) for x in val]) for key, val in base.items()}

    out = [base, mapv(lambda x: -x), mapv(lambda x: round(rnd.uniform(-4, 4), 3))]
    zeros = mapv(lambda x: x)
    for val in zeros.values():      # the first component of every vector zero
        for v in (val if isinstance(val[0], list) else [val]):
            v[0] = 0.0
    out.append(zeros)
    if name == "distances":
        out.append(dict(a=list(base["a"]), b=list(base["a"])))      # a == b: every hamming comparison ties
    else:
        key = "database" if name == "query" else "vectors"
        tied = mapv(lambda x: x)
        tied[key] = [list(tied[key][0]) for _ in tied[key]]
        out.append(tied)
    return out


def _host(Z, name, inp):
    """the host layout of inp, or the H2VError text"""
    try:
        return _example(Z, name, inp)
    except ValueError as e:
        return str(e)


# ----------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("name", ["distances", "query", "kmeans"])
def test_recording_builder_lays_out_the_same_circuit(name):
    Z = _Z()
    inp = Z.example_input(name)
    a, b = _example(Z, name, inp), _example(Z, name, inp, record=True)
    assert _layout_bytes(a) == _layout_bytes(b)
    ta, tb = a.builder.trace(), b.builder.trace()
    assert all((x == y).all() for x, y in zip(ta, tb))


@pytest.mark.parametrize("name", ["distances", "query", "kmeans"])
def test_cells_do_not_depend_on_the_input(name):
    Z = _Z()
    rec = _example(Z, name, Z.example_input(name), record=True)
    other = _example(Z, name, _variants(Z, name)[2])
    assert rec.break_points == other.break_points
    assert [c.tobytes() for c in rec.fixed] == [c.tobytes() for c in other.fixed]
    assert [c.tobytes() for c in rec.sigma] == [c.tobytes() for c in other.sigma]
    assert [c.tobytes() for c in rec.advice] != [c.tobytes() for c in other.advice]


@pytest.mark.parametrize("name", ["distances", "query", "kmeans"])
def test_program_inputs_and_info(name):
    Z = _Z()
    inp = Z.example_input(name)
    rc = _example(Z, name, inp, record=True)
    prog = Z.WitnessProgram(rc.builder, rc.k)
    want = Z.example_witness_inputs(name, inp)
    assert (prog.inputs() == want).all()
    info = prog.info
    assert info["inputs"] == len(want) == prog.n_inputs
    assert info["cells"] == rc.builder.stats()["advice_cells"]
    assert 0 < info["computed_cells"] < info["cells"]
    assert info["levels"] >= 1
    assert info["advice_columns"] == len(rc.advice) and info["instances"] == len(rc.instances[0]) and info["k"] == rc.k
    assert sum(prog.rule_counts()) == info["computed_cells"]
    rc.builder.close()      # the program owns what it needs
    assert (prog.inputs() == want).all()


def test_argument_errors_come_before_device_work():
    Z = _Z()
    from halo2_vectordb_b200 import lib

    rc = _example(Z, "distances", Z.example_input("distances"), record=True)
    prog = Z.WitnessProgram(rc.builder, rc.k)
    L, n = lib(), prog.n_inputs
    good = np.ascontiguousarray(prog.inputs()[None])
    adv = np.zeros((1, prog.info["advice_columns"], 1 << rc.k, 4), dtype=np.uint64)
    inst = np.zeros((1, prog.info["instances"], 4), dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.h2v_witness_generate(prog._h, 0, n, None, None, None) == 0
    assert L.h2v_witness_generate(None, 1, n, p(good), p(adv), p(inst)) == -1
    assert L.h2v_witness_generate(prog._h, 1, n + 1, p(good), p(adv), p(inst)) == -1
    assert L.h2v_witness_generate(prog._h, 1, n, None, p(adv), p(inst)) == -1
    assert L.h2v_witness_generate(prog._h, 1, n, p(good), None, p(inst)) == -1
    assert L.h2v_witness_generate(prog._h, 1, n, p(good), p(adv), None) == -1
    bad = good.copy()
    bad[0, 2] = [0xF0000001, 0, 0, 0x40000000_00000000]      # not below r
    assert L.h2v_witness_generate(prog._h, 1, n, p(bad), p(adv), p(inst)) == -1
    assert b"witness 0: input 2 is not a reduced Montgomery value" in L.h2v_last_error()
    if L.h2v_device_count() == 0:
        assert L.h2v_witness_generate(prog._h, 1, n, p(good), p(adv), p(inst)) == -2
    with pytest.raises(ValueError, match="not a recording builder"):
        Z.WitnessProgram(_example(Z, "distances", Z.example_input("distances")).builder, rc.k)


# ----------------------------------------------------------------------------------------------- GPU
def _check_equal(Z, prog, inputs, hosts):
    got = prog.generate(inputs)
    for w, ((adv, inst), rc) in enumerate(zip(got, hosts)):
        assert len(adv) == len(rc.advice)
        for c, (x, y) in enumerate(zip(adv, rc.advice)):
            assert x.tobytes() == y.tobytes(), f"witness {w}: advice column {c}"
        assert inst[0].tobytes() == rc.instances[0].tobytes(), f"witness {w}: instances"
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["distances", "query", "kmeans"])
def test_examples_byte_equal(h2v, name):
    Z = _Z()
    rec = _example(Z, name, Z.example_input(name), record=True)
    prog = Z.WitnessProgram(rec.builder, rec.k)
    pairs = [(v, _host(Z, name, v)) for v in _variants(Z, name)]
    pairs = [(v, rc) for v, rc in pairs if not isinstance(rc, str)]
    assert len(pairs) >= 4
    _check_equal(Z, prog, [Z.example_witness_inputs(name, v) for v, _ in pairs], [rc for _, rc in pairs])


K_OPS, LB_OPS = 13, 8
EDGE = [0, 1, R - 1, 2, R - 2, 1 << (2 * PREC), R - (1 << (2 * PREC)), R - (1 << (2 * PREC + 1)), R - (1 << (2 * PREC + 1)) + 1,
        R - (1 << (2 * PREC + 1)) - 1, 1 << PREC, R - (1 << PREC), 1 << (PREC - 1), 3 << PREC, R - (5 << (PREC - 2))]


def _op_cases():
    Z = _Z()
    unary = ["neg", "qabs", "is_neg", "sign", "clip", "qexp2", "qlog2", "qexp", "qlog", "qsqrt", "qsin", "qcos", "qtan", "qsinh",
             "qcosh", "qtanh"]
    binary = ["qadd", "qsub", "qmul", "qdiv", "qmod", "qpow", "qmax", "qmin", "bit_xor", "cond_neg"]
    cases = [(n, 1) for n in unary] + [(n, 2) for n in binary] + [("qsum", 4), ("inner_product", 4), ("polynomial", 4)]
    cases += [(d, 6) for d in ("euclidean", "cosine", "hamming", "manhattan")]
    cases += [("poseidon_hash", 3), ("merkle_commitment", 6)]
    return cases


def _record_op(Z, op, vals, record):
    """a small circuit: assign vals, apply op, make the result public"""
    b = Z.GateThreadBuilder(LB_OPS, PREC, record=record)
    ctx = b.main(0)
    fp = Z.FixedPointChip.default(b)
    cells = ctx.assign_witnesses(_mont(vals))
    if op in ("euclidean", "cosine", "hamming", "manhattan"):
        out = getattr(Z.DistanceChip.default(fp), op + "_distance")(ctx, cells[:3], cells[3:])
    elif op == "poseidon_hash":
        ph = Z.PoseidonChip(ctx, 8, 57)
        ph.update(cells)
        out = ph.squeeze(ctx)
    elif op == "merkle_commitment":
        ph = Z.PoseidonChip(ctx, 8, 57)
        out = Z.VectorDBChip.default(fp).merkle_commitment(ctx, ph, [cells[:2], cells[2:4], cells[4:]])
    elif op == "qsum":
        out = fp.qsum(ctx, cells)
    elif op == "inner_product":
        out = fp.inner_product(ctx, cells[:2], cells[2:])
    elif op == "polynomial":
        out = fp.polynomial(ctx, cells[0], cells[1:])
    else:
        out = getattr(fp, op)(ctx, *cells)
    b.make_public([out])
    return Z.RangeCircuit(b, K_OPS)


def _mont(vals):
    from common import fr_arr

    return fr_arr([v % R for v in vals])


def _op_inputs(arity, seed):
    rnd = random.Random(seed)
    q = lambda: round(rnd.uniform(-6, 6), 4)
    quant = lambda x: int(round(abs(x) * (1 << PREC))) * (1 if x >= 0 else -1)
    rows = [[EDGE[(i + j) % len(EDGE)] for j in range(arity)] for i in range(len(EDGE))]
    rows += [[quant(q()) for _ in range(arity)] for _ in range(6)]
    rows.append([1 << PREC] * arity)      # a divisor of 1
    return [[v % R for v in r] for r in rows]


@pytest.mark.gpu
def test_ops_byte_equal(h2v):
    Z = _Z()
    kinds = None
    for i, (op, arity) in enumerate(_op_cases()):
        rows = _op_inputs(arity, i)
        rec = _record_op(Z, op, [(1 + j) << PREC for j in range(arity)], record=True)
        prog = Z.WitnessProgram(rec.builder, K_OPS)
        counts = np.array(prog.rule_counts())
        kinds = counts if kinds is None else kinds + counts
        ok, failing = [], []
        for r in rows:
            try:
                ok.append((r, _record_op(Z, op, r, record=False)))
            except ValueError as e:
                failing.append((r, str(e)))
        for rc in [rc for _, rc in ok]:
            assert rc.break_points == rec.break_points, op
        if ok:
            _check_equal(Z, prog, [_mont(r) for r, _ in ok], [rc for _, rc in ok])
        for r, text in failing:      # the host panics: so does the replay, with the host's text
            with pytest.raises(ValueError, match="witness 0: " + text.split(":")[-1].strip()):
                prog.generate([_mont(r)])
    assert all(kinds[4:] > 0), f"rule kinds never computed: {[k for k in range(4, len(kinds)) if not kinds[k]]}"


@pytest.mark.gpu
def test_division_by_zero_names_the_lowest_witness(h2v):
    Z = _Z()
    rec = _record_op(Z, "qdiv", [5 << PREC, 2 << PREC], record=True)
    prog = Z.WitnessProgram(rec.builder, K_OPS)
    good = [[(w + 1) << PREC, (w + 2) << PREC] for w in range(6)]
    bad = [list(r) for r in good]
    bad[2][1] = bad[4][1] = 0
    with pytest.raises(ValueError, match=r"witness_generate: witness 2: attempt to divide by zero \(cell \d+\)"):
        prog.generate([_mont(r) for r in bad])
    _check_equal(Z, prog, [_mont(r) for r in good], [_record_op(Z, "qdiv", r, record=False) for r in good])


@pytest.mark.gpu
def test_group_sizes_give_the_same_bytes(h2v, monkeypatch):
    Z = _Z()
    name = "query"
    rec = _example(Z, name, Z.example_input(name), record=True)
    prog = Z.WitnessProgram(rec.builder, rec.k)
    inputs = [Z.example_witness_inputs(name, v) for v in _variants(Z, name)[:3]]
    one = prog.generate(inputs)
    for g in ("1", "2"):
        monkeypatch.setenv("H2V_PROOF_GROUP", g)
        got = prog.generate(inputs)
        assert [[c.tobytes() for c in a] + [i[0].tobytes()] for a, i in got] == [[c.tobytes() for c in a] + [i[0].tobytes()] for a, i in one]
    assert prog.generate([]) == []


def _untied_query(Z, shift):
    inp = Z.example_input("query")
    inp["database"] = [[x + 1e-3 * (i // 4) + shift for x in v] for i, v in enumerate(inp["database"])]
    return inp


@pytest.mark.gpu
def test_generated_columns_prove_and_check(h2v):
    Z = _Z()
    ins = [_untied_query(Z, s) for s in (0.0, 0.25, -0.5, 1.0)]
    rec = _example(Z, "query", ins[0], record=True)
    prog = Z.WitnessProgram(rec.builder, rec.k)
    hosts = [_example(Z, "query", v) for v in ins]
    gen = _check_equal(Z, prog, [Z.example_witness_inputs("query", v) for v in ins], hosts)
    srs = h2v.ParamsKZG.gen_srs(rec.k)
    pk = h2v.ProvingKey(srs, rec.cs, rec.fixed, rec.sigma, np.array([rec.k, 0, 0, 0], dtype=np.uint64))
    seeds = [bytes([p]) * 32 for p in range(4)]
    want = pk.create_proofs([rc.advice for rc in hosts], [rc.instances for rc in hosts], seeds)
    assert pk.create_proofs([a for a, _ in gen], [i for _, i in gen], seeds) == want
    assert [m.n_failures for m in pk.mock_prover([a for a, _ in gen], [i for _, i in gen])] == [0] * 4
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_unsatisfied_qlog2_gives_the_host_failures(h2v):
    Z = _Z()
    rec = _record_op(Z, "qlog2", [3 << PREC], record=True)
    prog = Z.WitnessProgram(rec.builder, K_OPS)
    rows = [[R - (3 << PREC)], [0]]
    hosts = [_record_op(Z, "qlog2", r, record=False) for r in rows]
    gen = _check_equal(Z, prog, [_mont(r) for r in rows], hosts)
    srs = h2v.ParamsKZG.gen_srs(K_OPS)
    pk = h2v.ProvingKey(srs, rec.cs, rec.fixed, rec.sigma, np.array([K_OPS, 0, 0, 0], dtype=np.uint64))
    got = pk.mock_prover([a for a, _ in gen], [i for _, i in gen])
    want = pk.mock_prover([rc.advice for rc in hosts], [rc.instances for rc in hosts])
    for g, w in zip(got, want):
        assert g.n_failures > 0
        assert g.n_failures == w.n_failures and g.failures == w.failures
    pk.close()
    srs.close()
