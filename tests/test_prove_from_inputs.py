"""Proofs and mock checks straight from inputs (h2v_create_proofs_from_inputs, h2v_pk_mock_prover_from_inputs): the
witness program's columns are generated in the key's workspace, and the results must equal, byte for byte, those of
h2v_witness_generate followed by h2v_create_proofs / h2v_pk_mock_prover with the same seeds."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import pyref as P

R = P.R
PREC = 48
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CALLS = ["h2v_create_proofs_from_inputs", "h2v_pk_mock_prover_from_inputs"]


def _Z():
    from halo2_vectordb_b200 import circuit as Z

    return Z


def _record(Z, name, inp):
    k, bits = Z.EXAMPLE_PARAMS[name]
    return Z.create_circuit(Z.EXAMPLES[name], inp, k, bits, record=True)[0]


def _untied_query(Z, shift):
    """data/query.in with its five-way distance ties broken, shifted"""
    inp = Z.example_input("query")
    inp["database"] = [[x + 1e-3 * (i // 4) + shift for x in v] for i, v in enumerate(inp["database"])]
    return inp


def _shifted(Z, name, shift):
    """the example input with every value moved by shift (the recording's shape)"""
    return {key: ([[x + shift for x in v] for v in val] if isinstance(val[0], list) else [x + shift for x in val])
            for key, val in Z.example_input(name).items()}


def _inputs(Z, name, B):
    if name == "query":
        ins = [_untied_query(Z, s) for s in (0.0, 0.25, -0.5, 1.0, 0.125)[:B]]
    else:
        ins = [_shifted(Z, name, s) for s in (0.0, 0.25, -0.5, 1.0, 0.125)[:B]]
    return ins


def _mont(vals):
    from common import fr_arr

    return fr_arr([v % R for v in vals])


def _record_op(Z, op, vals, k=13):
    """a small recorded circuit: assign vals, apply the FixedPointChip op, make the result public"""
    b = Z.GateThreadBuilder(8, PREC, record=True)
    ctx = b.main(0)
    fp = Z.FixedPointChip.default(b)
    cells = ctx.assign_witnesses(_mont(vals))
    b.make_public([getattr(fp, op)(ctx, *cells)])
    return Z.RangeCircuit(b, k)


class Case:
    """a recording, its program and a key loaded from its layout"""

    def __init__(self, h, rec):
        self.rec = rec
        self.prog = _Z().WitnessProgram(rec.builder, rec.k)
        self.srs = h.ParamsKZG.gen_srs(rec.k)
        self.pk = self.key(h)

    def key(self, h):
        rec = self.rec
        return h.ProvingKey(self.srs, rec.cs, rec.fixed, rec.sigma, np.array([rec.k, 0, 0, 0], dtype=np.uint64))

    def reference(self, inputs, seeds, pk=None):
        """generate -> create_proofs: (proofs, instances)"""
        gen = self.prog.generate(inputs)
        return (pk or self.pk).create_proofs([a for a, _ in gen], [i for _, i in gen], seeds), [i for _, i in gen]


_CASES = {}


@pytest.fixture
def case(h2v):
    def get(name):
        if name not in _CASES:
            Z = _Z()
            _CASES[name] = Case(h2v, _record(Z, name, _inputs(Z, name, 1)[0]))
        return _CASES[name]

    return get


def _seeds(B, salt=0):
    return [bytes([p + salt]) * 32 for p in range(B)]


def _same_instances(got, want):
    assert [[c.tobytes() for c in g] for g in got] == [[c.tobytes() for c in w] for w in want]


# ----------------------------------------------------------------------------------------------- no device needed
def test_symbols_declared_and_exported():
    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import build

    build.build()
    hdr = open(os.path.join(ROOT, "include", "h2v.h")).read()
    hpp = open(os.path.join(ROOT, "include", "h2v.hpp")).read()
    rs = open(os.path.join(ROOT, "ffi", "src", "lib.rs")).read()
    for name in CALLS:
        assert re.search(r"\bint " + name + r"\s*\(", hdr), name
        assert name in h.ABI_SYMBOLS and hasattr(h.lib(), name), name
        assert name in hpp and "pub fn " + name in rs, name
    assert "create_proofs_from_inputs" in rs and "mock_prover_from_inputs" in rs


def test_null_handles_and_empty_batches():
    from halo2_vectordb_b200 import lib

    Z = _Z()
    rec = _record(Z, "distances", Z.example_input("distances"))
    prog = Z.WitnessProgram(rec.builder, rec.k)
    L, n = lib(), prog.n_inputs
    good = np.ascontiguousarray(prog.inputs()[None])
    seeds = bytes(32)
    out = np.zeros(1 << 16, dtype=np.uint8)
    totals = np.zeros(1, dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.h2v_create_proofs_from_inputs(None, prog._h, 1, n, p(good), seeds, p(out), out.size, None) == -1
    assert L.h2v_last_error().startswith(b"create_proofs_from_inputs: NULL key")
    assert L.h2v_pk_mock_prover_from_inputs(None, prog._h, 1, n, p(good), None, 0, p(totals)) == -1
    assert L.h2v_last_error().startswith(b"pk_mock_prover_from_inputs: NULL key")
    # a key handle is not read when the batch is empty or the program is missing: any non-NULL value stands for one here
    fake_key = C.c_void_p(out.ctypes.data)
    assert L.h2v_create_proofs_from_inputs(fake_key, None, 1, n, p(good), seeds, p(out), out.size, None) == -1
    assert L.h2v_last_error().startswith(b"create_proofs_from_inputs: NULL key or program")
    assert L.h2v_pk_mock_prover_from_inputs(fake_key, None, 1, n, p(good), None, 0, p(totals)) == -1
    assert L.h2v_last_error().startswith(b"pk_mock_prover_from_inputs: NULL key or program")
    assert L.h2v_create_proofs_from_inputs(fake_key, prog._h, 0, n, None, None, None, 0, None) == 0
    assert L.h2v_pk_mock_prover_from_inputs(fake_key, prog._h, 0, n, None, None, 0, None) == 0


# ----------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("distances", 5), ("query", 5), ("kmeans", 2)])
def test_proofs_equal_generate_then_create_proofs(h2v, case, name, B):
    c = case(name)
    inputs = [_Z().example_witness_inputs(name, v) for v in _inputs(_Z(), name, B)]
    seeds = _seeds(B)
    want, want_inst = c.reference(inputs, seeds)
    got, inst = c.pk.create_proofs_from_inputs(c.prog, inputs, seeds)
    assert got == want
    _same_instances(inst, want_inst)
    ms = c.pk.last_phase_ms()
    assert ms["advice_commit"] > 0
    assert all(t >= 0 for t in c.prog.last_ms()) and c.prog.last_ms()[1] > 0
    assert c.pk.create_proofs_from_inputs(c.prog, [], []) == ([], [])


@pytest.mark.gpu
def test_group_sizes_and_streamed_key_give_the_same_bytes(h2v, case, monkeypatch):
    c = case("query")
    Z = _Z()
    inputs = [Z.example_witness_inputs("query", v) for v in _inputs(Z, "query", 5)]
    seeds = _seeds(5, salt=9)
    want, want_inst = c.reference(inputs, seeds)
    for g in ("1", "2", "3"):
        monkeypatch.setenv("H2V_PROOF_GROUP", g)
        got, inst = c.pk.create_proofs_from_inputs(c.prog, inputs, seeds)
        assert got == want, g
        _same_instances(inst, want_inst)
        assert c.pk.last_phase_ms()["advice_commit"] > 0
    monkeypatch.delenv("H2V_PROOF_GROUP")
    monkeypatch.setenv("H2V_STREAM_EXT", "1")
    pk = c.key(h2v)
    assert pk.create_proofs_from_inputs(c.prog, inputs[:2], seeds[:2])[0] == want[:2]
    pk.close()


@pytest.mark.gpu
def test_a_panicking_witness_is_named_and_leaves_key_and_program_usable(h2v):
    Z = _Z()
    rec = _record_op(Z, "qdiv", [5 << PREC, 2 << PREC])
    c = Case(h2v, rec)
    good = [_mont([(w + 1) << PREC, (w + 2) << PREC]) for w in range(6)]
    bad = list(good)
    bad[2] = bad[4] = _mont([3 << PREC, 0])
    seeds = _seeds(6)
    with pytest.raises(ValueError, match=r"^create_proofs_from_inputs: witness 2: attempt to divide by zero \(cell \d+\)"):
        c.pk.create_proofs_from_inputs(c.prog, bad, seeds)
    with pytest.raises(ValueError, match=r"^pk_mock_prover_from_inputs: witness 2: attempt to divide by zero \(cell \d+\)"):
        c.pk.mock_prover_from_inputs(c.prog, bad)
    want, want_inst = c.reference(good, seeds)
    got, inst = c.pk.create_proofs_from_inputs(c.prog, good, seeds)
    assert got == want
    _same_instances(inst, want_inst)
    assert [m.n_failures for m in c.pk.mock_prover_from_inputs(c.prog, good)] == [0] * 6
    c.pk.close()
    c.srs.close()


@pytest.mark.gpu
def test_mismatched_program_is_refused_before_device_work(h2v, case):
    Z = _Z()
    q, d = case("query"), case("distances")
    assert q.rec.k == d.rec.k and q.prog.info["advice_columns"] != d.prog.info["advice_columns"]
    inputs = [Z.example_witness_inputs("distances", Z.example_input("distances"))]
    launches = h2v.launch_count()
    with pytest.raises(ValueError, match=r"^create_proofs_from_inputs: the program has \d+ advice columns, the key \d+"):
        q.pk.create_proofs_from_inputs(d.prog, inputs, _seeds(1))
    with pytest.raises(ValueError, match=r"^pk_mock_prover_from_inputs: the program has \d+ advice columns"):
        q.pk.mock_prover_from_inputs(d.prog, inputs)
    bad = np.array(inputs[0], dtype=np.uint64)
    bad[1] = [0xF0000001, 0, 0, 0x40000000_00000000]      # not below r
    with pytest.raises(ValueError, match="witness 0: input 1 is not a reduced Montgomery value"):
        d.pk.create_proofs_from_inputs(d.prog, [bad], _seeds(1))
    L = h2v.lib()
    size = d.pk.proof_size()
    out = np.zeros(size, dtype=np.uint8)
    good = np.ascontiguousarray(inputs[0])
    assert L.h2v_create_proofs_from_inputs(d.pk._h, d.prog._h, 1, d.prog.n_inputs + 1, good.ctypes.data, bytes(32), out.ctypes.data, size,
                                           None) == -1
    assert b"inputs per witness" in L.h2v_last_error()
    assert L.h2v_create_proofs_from_inputs(d.pk._h, d.prog._h, 1, d.prog.n_inputs, good.ctypes.data, bytes(32), out.ctypes.data, size - 1,
                                           None) == -1
    assert b"proof_stride" in L.h2v_last_error()
    assert h2v.launch_count() == launches


@pytest.mark.gpu
def test_mock_equals_pk_mock_prover_on_generated_columns(h2v, case):
    Z = _Z()
    # data/query.in as recorded: its five-way ties give 12 gate failures
    rec = _record(Z, "query", Z.example_input("query"))
    c = Case(h2v, rec)
    inputs = [c.prog.inputs()] * 2
    gen = c.prog.generate(inputs)
    want = c.pk.mock_prover([a for a, _ in gen], [i for _, i in gen])
    got = c.pk.mock_prover_from_inputs(c.prog, inputs)
    assert [(m.failures, m.n_failures) for m in got] == [(m.failures, m.n_failures) for m in want]
    assert all(m.n_failures == 12 and all(f.kind == h2v.MOCK_GATE for f in m.failures) for m in got)
    assert got[0].upload_ms > 0
    c.pk.close()
    c.srs.close()
    # the untied query: satisfied
    q = case("query")
    ins = [Z.example_witness_inputs("query", v) for v in _inputs(Z, "query", 3)]
    assert [m.n_failures for m in q.pk.mock_prover_from_inputs(q.prog, ins)] == [0] * 3
    # qlog2 on -3 and 0: unsatisfied, the host's failures
    rec = _record_op(Z, "qlog2", [3 << PREC])
    c = Case(h2v, rec)
    rows = [_mont([R - (3 << PREC)]), _mont([0])]
    gen = c.prog.generate(rows)
    want = c.pk.mock_prover([a for a, _ in gen], [i for _, i in gen], max_failures=8)
    got = c.pk.mock_prover_from_inputs(c.prog, rows, max_failures=8)
    assert all(m.n_failures > 0 for m in got)
    assert [(m.failures, m.n_failures) for m in got] == [(m.failures, m.n_failures) for m in want]
    c.pk.close()
    c.srs.close()


@pytest.mark.gpu
def test_proof_after_mock_call_equals_a_fresh_keys(h2v, case):
    Z = _Z()
    q = case("query")
    ins = [Z.example_witness_inputs("query", v) for v in _inputs(Z, "query", 3)]
    seeds = _seeds(3, salt=40)
    q.pk.mock_prover_from_inputs(q.prog, ins[::-1])
    got, _ = q.pk.create_proofs_from_inputs(q.prog, ins, seeds)
    fresh = q.key(h2v)
    assert got == fresh.create_proofs_from_inputs(q.prog, ins, seeds)[0]
    fresh.close()


@pytest.mark.gpu
def test_two_devices(h2v):
    if h2v.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    Z = _Z()
    rec = _record(Z, "query", _inputs(Z, "query", 1)[0])
    ins = [Z.example_witness_inputs("query", v) for v in _inputs(Z, "query", 4)]
    seeds = _seeds(4, salt=3)
    results = []
    try:
        for devs in ([0], [0, 1]):
            h2v.init(devs)
            c = Case(h2v, rec)
            results.append(c.pk.create_proofs_from_inputs(c.prog, ins, seeds)[0])
            c.pk.close()
            c.srs.close()
            c.prog.close()
    finally:
        h2v.init(0)
    assert results[0] == results[1]
