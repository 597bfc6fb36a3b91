"""h2v_mock_prover: halo2's MockProver checks (gates, lookups, copy constraints) on the device.

The specification is oracle/mock.py::mock_prover: wherever it can run, the device's failure list, formatted into the
oracle's messages with the host columns, must equal the oracle's list entry for entry (same order, same cap).  Where it
cannot (kmeans at k = 16, a k = 18 circuit), the satisfied layout must give no failure and a seeded change must give
exactly the failures derived here from the columns near the changed cells."""
import copy
import ctypes as C

import numpy as np
import pytest

from common import fr_arr
from oracle import mock as M
from oracle import oracle as O
from oracle import pyref as P
from toy_circuit import Toy

R = P.R
DELTA = pow(P.GEN, 1 << P.S, R)
BIG = 1 << 30                   # "no cap" for the oracle


@pytest.fixture(scope="module")
def Z():
    from halo2_vectordb_b200 import circuit as z

    return z


# ----------------------------------------------------------------------------------------------- helpers
def _ints(cols):
    return [O.fr_to_ints(np.ascontiguousarray(c)) for c in cols]


def _messages(h, cs, fails, fixed, advice, instances):
    """the oracle's message for each failure, values read from the host columns (lists of canonical ints)"""
    n = 1 << cs["k"]

    def cell(c, r):
        kind, idx = cs["permutation"][c]
        if kind == 0:
            return advice[idx][r]
        if kind == 1:
            return fixed[idx][r]
        return instances[idx][r] if r < len(instances[idx]) else 0

    out = []
    for f in fails:
        if f.kind == h.MOCK_GATE:
            out.append(f"gate not satisfied: column {f.other_column} row {f.row}")
        elif f.kind == h.MOCK_GATE_UNUSABLE:
            out.append(f"gate on column {f.other_column} row {f.row} reaches into the unusable rows")
        elif f.kind == h.MOCK_LOOKUP:
            out.append(f"lookup: column {f.other_column} row {f.row} holds {advice[f.other_column][f.row]}, not in the table")
        elif f.kind == h.MOCK_SIGMA_NOT_DELTA_OMEGA:
            assert (f.other_column, f.other_row) == (0xFFFFFFFF, 0xFFFFFFFF)
            out.append(f"sigma column {f.column} row {f.row} is not delta^i omega^j")
        elif f.kind == h.MOCK_SIGMA_NOT_PERMUTATION:
            out.append(f"sigma is not a permutation: ({f.other_column}, {f.other_row}) hit twice")
        elif f.kind == h.MOCK_COPY_UNUSABLE:
            out.append(f"copy constraint touches an unusable row: ({f.column}, {f.row}) -> ({f.other_column}, {f.other_row})")
        elif f.kind == h.MOCK_COPY:
            out.append(f"copy constraint violated: ({f.column}, {f.row}) = {cell(f.column, f.row)} vs "
                       f"({f.other_column}, {f.other_row}) = {cell(f.other_column, f.other_row)}")
        else:
            raise AssertionError(f"unknown kind {f.kind}")
        assert f.row < n
    return out


def _check_ints(h, cs, fixed, sigma, advice, instances, cap=BIG):
    """device vs oracle on columns of canonical ints; returns the oracle's list"""
    want = M.mock_prover(cs, fixed, sigma, advice, instances, max_failures=cap)
    mp = h.MockProver.run(cs, [fr_arr(c) for c in fixed], [fr_arr(c) for c in sigma], [fr_arr(c) for c in advice],
                          [fr_arr(c) for c in instances], max_failures=min(cap, 4096))
    assert _messages(h, cs, mp.failures, fixed, advice, instances) == want
    if cap == BIG:
        assert mp.n_failures == len(want)
    return want, mp


def _toy_check(h, t, cap=BIG):
    return _check_ints(h, t.cs, t.fixed, t.sigma, t.advice, t.instances, cap)


# ----------------------------------------------------------------------------------------------- toy circuits
TOYS = [(6, 1, 2, 1), (7, 2, 3, 2), (8, 3, 1, 1), (9, 4, 4, 0), (10, 5, 2, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("k,seed,gate_cols,lookup_cols", TOYS)
def test_toy_honest_and_broken(h2v, k, seed, gate_cols, lookup_cols):
    t = Toy(k, seed=seed, n_gate_cols=gate_cols, n_lookup_cols=lookup_cols)
    want, mp = _toy_check(h2v, t)
    assert want == [] and mp.failures == [] and mp.n_failures == 0
    mp.assert_satisfied()
    for how in ("break_gate", "break_copy", "break_public_input"):
        w = copy.deepcopy(t)
        getattr(w, how)()
        want, mp = _toy_check(h2v, w)
        assert want, how
        with pytest.raises(AssertionError, match="not satisfied"):
            mp.assert_satisfied()


@pytest.mark.gpu
def test_toy_unreduced_limbs_are_field_elements(h2v):
    """value + r (limbs above the modulus) is the same field element: no failure"""
    t = Toy(7, seed=3, n_gate_cols=2, n_lookup_cols=1)
    n = 1 << 7

    def unreduce(col):
        raw = O.limbs_to_ints(col)
        return O.ints_to_limbs([x + R if x + R < 1 << 256 else x for x in raw])

    adv = [unreduce(fr_arr(c)) for c in t.advice]
    fixed = [unreduce(fr_arr(c)) for c in t.fixed]
    sigma = [unreduce(fr_arr(c)) for c in t.sigma]
    assert sum(int((a != fr_arr(c)).any(axis=1).sum()) for a, c in zip(adv, t.advice)) > n
    mp = h2v.MockProver.run(t.cs, fixed, sigma, adv, [unreduce(fr_arr(c)) for c in t.instances])
    assert mp.n_failures == 0 and mp.failures == []


@pytest.mark.gpu
@pytest.mark.parametrize("fault", ["swap", "not_delta_omega", "duplicate", "selector_in_blinding_rows", "copy_into_unusable"])
def test_hand_made_key_faults(h2v, fault):
    t = Toy(8, seed=17, n_gate_cols=3, n_lookup_cols=2)
    n, u = t.n, t.u
    omega = P.omega_for(t.k)
    pc = t.cs["permutation"].index((0, 0))      # the permutation column of advice column 0
    if fault == "swap":
        t.sigma[pc][1], t.sigma[pc][6] = t.sigma[pc][6], t.sigma[pc][1]
    elif fault == "not_delta_omega":
        t.sigma[pc + 1][5] = 12345
        t.sigma[pc][0] = 0
    elif fault == "duplicate":
        t.sigma[pc][9] = t.sigma[pc][10]
    elif fault == "selector_in_blinding_rows":
        t.fixed[0][n - 2] = 1
        t.fixed[1][u - 2] = 5
    elif fault == "copy_into_unusable":
        old = t.sigma[pc][2]
        t.sigma[pc][2] = pow(DELTA, pc, R) * pow(omega, n - 1, R) % R
        t.sigma[pc][n - 1] = old
    want, mp = _toy_check(h2v, t)
    assert want
    # the cap: the first entries of the same list, and the exact total
    for cap in {1, 2, max(1, len(want) - 1)}:
        mp2 = h2v.MockProver.run(t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], [fr_arr(c) for c in t.advice],
                                 [fr_arr(c) for c in t.instances], max_failures=cap)
        assert mp2.failures == mp.failures[:cap] and mp2.n_failures == len(want)


# ----------------------------------------------------------------------------------------------- the examples
def _layout(Z, name, inp=None):
    k0, lb0 = Z.EXAMPLE_PARAMS[name]
    return Z.create_circuit(Z.EXAMPLES[name], inp or Z.example_input(name), k0, lb0)


@pytest.mark.gpu
def test_distances_example(h2v, Z):
    rc, _ = _layout(Z, "distances")
    fixed, sigma, advice, inst = _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances)
    mp = h2v.MockProver.run(rc.cs, rc.fixed, rc.sigma, rc.advice, rc.instances)
    assert mp.failures == [] and mp.n_failures == 0
    bad = [list(c) for c in advice]
    bad[0][7] = (bad[0][7] + 1) % R
    want, _ = _check_ints(h2v, rc.cs, fixed, sigma, bad, inst)
    assert len(want) >= 2
    want, _ = _check_ints(h2v, rc.cs, fixed, sigma, advice, [[(inst[0][0] + 1) % R] + inst[0][1:]])
    assert want
    bad = [list(c) for c in advice]
    bad[rc.num_advice][3] = 1 << 12
    bad[rc.num_advice + 1][20] = R - 1
    want, mp = _check_ints(h2v, rc.cs, fixed, sigma, bad, inst)
    assert sum(f.kind == h2v.MOCK_LOOKUP for f in mp.failures) == 2
    # cap below the total: the first `cap` entries of the oracle's capped list, the oracle's uncapped count
    for cap in (1, 3, len(want) - 1):
        got, mp = _check_ints(h2v, rc.cs, fixed, sigma, bad, inst, cap=cap)
        assert len(got) == cap and mp.n_failures == len(want)


@pytest.mark.gpu
def test_query_example(h2v, Z):
    rc, _ = _layout(Z, "query")
    want, mp = _check_ints(h2v, rc.cs, _ints(rc.fixed), _ints(rc.sigma), _ints(rc.advice), _ints(rc.instances))
    assert len(want) == 12 and all(f.kind == h2v.MOCK_GATE for f in mp.failures)
    inp = Z.example_input("query")
    inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
    rc, _ = _layout(Z, "query", inp=inp)
    mp = h2v.MockProver.run(rc.cs, rc.fixed, rc.sigma, rc.advice, rc.instances)
    assert mp.failures == [] and mp.n_failures == 0


# ----------------------------------------------------------------------------------------------- too large for the oracle
def _expected(h, cs, fixed, sigma, advice, instances, changed):
    """The failures a change of the advice cells `changed` [(column, row)] causes in a circuit that was satisfied, by the
    oracle's rules applied to the cells near them: the <= 4 gate rows that read each cell, each lookup of its column, and
    the cell's successor and predecessor in its copy cycle (found by decoding sigma along the cycle)."""
    k = cs["k"]
    n, u = 1 << k, (1 << k) - cs["blinding_factors"] - 1
    val = lambda col, r: O.fr_to_ints(np.ascontiguousarray(col[r:r + 1]))[0]
    perm = cs["permutation"]

    def cell(c, r):
        kind, idx = perm[c]
        if kind == 2:
            return val(instances[idx], r) if r < len(instances[idx]) else 0
        return val((advice, fixed)[kind][idx], r)

    gates, lookups, copies = [], [], set()
    for j, (a, q) in enumerate(cs["gates"]):
        for s in sorted({s for c, r in changed if c == a for s in range(max(0, r - 3), r + 1)}):
            if val(fixed[q], s):
                assert s + 3 < u
                x = [val(advice[a], s + i) for i in range(4)]
                if (x[0] + x[1] * x[2] - x[3]) % R:
                    gates.append((h.MOCK_GATE, j, s, a, s))
    tables = {}
    for l, (a, t) in enumerate(cs["lookups"]):
        if t not in tables:
            tables[t] = set(O.fr_to_ints(np.ascontiguousarray(fixed[t][:u])))
        for c, r in sorted(changed):
            if c == a and r < u and val(advice[a], r) not in tables[t]:
                lookups.append((h.MOCK_LOOKUP, l, r, a, r))
    col_of = {pow(pow(DELTA, c, R), n, R): c for c in range(len(perm))}
    omega = P.omega_for(k)
    row_of, w = {}, 1
    for r in range(n):
        row_of[w] = r
        w = w * omega % R

    dinv = [pow(pow(DELTA, c, R), R - 2, R) for c in range(len(perm))]

    def image(c, r):
        v = val(sigma[c], r)
        c2 = col_of[pow(v, n, R)]
        return c2, row_of[v * dinv[c2] % R]

    for a, r in changed:
        pc = perm.index((0, a))
        nxt = image(pc, r)
        if nxt == (pc, r):
            continue
        prev = nxt
        while (step := image(*prev)) != (pc, r):
            prev = step
        for x, y in (((pc, r), nxt), (prev, (pc, r))):
            if cell(*x) != cell(*y):
                copies.add((h.MOCK_COPY, x[0], x[1], y[0], y[1]))
    return gates + lookups + sorted(copies, key=lambda f: (f[1], f[2]))


def _change(h, rc_cs, fixed, sigma, advice, instances, changes):
    """advice[c][r] <- value for (c, r, value) in changes; the device's list must equal _expected's"""
    for c, r, v in changes:
        advice[c] = advice[c].copy()
        advice[c][r] = fr_arr([v])[0]
    want = _expected(h, rc_cs, fixed, sigma, advice, instances, [(c, r) for c, r, _ in changes])
    mp = h.MockProver.run(rc_cs, fixed, sigma, advice, instances, max_failures=256)
    assert [tuple(f) for f in mp.failures] == want and mp.n_failures == len(want)
    return want


@pytest.mark.gpu
def test_kmeans_example(h2v, Z):
    rc, _ = _layout(Z, "kmeans")
    assert (rc.num_advice, rc.num_lookup_advice) == (535, 72)
    mp = h2v.MockProver.run(rc.cs, rc.fixed, rc.sigma, rc.advice, rc.instances)
    assert mp.failures == [] and mp.n_failures == 0
    advice = list(rc.advice)
    j = 3
    a, q = rc.cs["gates"][j]
    sel = O.fr_to_ints(np.ascontiguousarray(rc.fixed[q][1000:2000]))
    r = 1000 + next(i for i, v in enumerate(sel) if v)  # the first cell of an enabled gate row: its gate must fail
    la, lr = rc.num_advice, 77                          # a lookup-column cell, moved outside the 2^15-value table
    old = O.fr_to_ints(np.ascontiguousarray(advice[a][r:r + 1]))[0]
    want = _change(h2v, rc.cs, rc.fixed, rc.sigma, advice, rc.instances, [(a, r, old + 1), (la, lr, 1 << 15)])
    kinds = {f[0] for f in want}
    assert h2v.MOCK_GATE in kinds and h2v.MOCK_LOOKUP in kinds


@pytest.mark.gpu
def test_large_k_synthetic_circuit(h2v):
    """k = 18: a satisfied Toy circuit gives no failure; one changed cell is found at its gate row and copy cells"""
    t = Toy(18, seed=5, n_gate_cols=2, n_lookup_cols=1, n_public=3)
    fixed, sigma, advice, inst = ([fr_arr(c) for c in cols] for cols in (t.fixed, t.sigma, t.advice, t.instances))
    mp = h2v.MockProver.run(t.cs, fixed, sigma, advice, inst)
    assert mp.failures == [] and mp.n_failures == 0
    r = 4 * 40000 + 2                                   # the c of gate row 160000 in gate column 1
    want = _change(h2v, t.cs, fixed, sigma, advice, inst, [(1, r, t.advice[1][r] + 1)])
    assert want[0] == (h2v.MOCK_GATE, 1, r - 2, 1, r - 2)


# ----------------------------------------------------------------------------------------------- input checks (no device needed)
def _raw_call(h, cs, fixed, sigma, advice, instances, inst_len=None, null=None):
    """h2v_mock_prover through ctypes, with one column list entry replaced by NULL"""
    ct, keep = h._circuit_struct(cs)
    lists = {"fixed": list(fixed), "sigma": list(sigma), "advice": list(advice), "instances": list(instances)}
    arrs = {}
    for name, cols in lists.items():
        ptrs = [c.ctypes.data for c in cols]
        if null and null[0] == name:
            ptrs[null[1]] = None
        arrs[name] = (C.c_void_p * max(1, len(ptrs)))(*ptrs)
    il = np.ascontiguousarray(inst_len if inst_len is not None else [c.shape[0] for c in instances], dtype=np.uint32)
    out = (h._MockFailureT * 4)()
    total = C.c_uint64()
    rc = h.lib().h2v_mock_prover(C.byref(ct), arrs["fixed"], arrs["sigma"], arrs["advice"], arrs["instances"],
                                 il.ctypes.data_as(C.c_void_p), out, 4, C.byref(total))
    return rc, h.lib().h2v_last_error().decode()


def test_invalid_inputs_are_rejected():
    import halo2_vectordb_b200 as h

    t = Toy(6, seed=2)
    n = t.n
    cols = [[fr_arr(c) for c in x] for x in (t.fixed, t.sigma, t.advice, t.instances)]
    with pytest.raises(ValueError, match="column count"):
        h.MockProver.run(t.cs, cols[0][:-1], *cols[1:])
    with pytest.raises(ValueError, match="column count"):
        h.MockProver.run(t.cs, cols[0], cols[1], cols[2] + cols[2][:1], cols[3])
    for null in (("fixed", 1), ("sigma", 0), ("advice", 2)):
        rc, msg = _raw_call(h, t.cs, *cols, null=null)
        assert rc == -1 and "NULL" in msg and null[0] in msg
    rc, msg = _raw_call(h, t.cs, *cols, inst_len=[n + 1])
    assert rc == -1 and "instance column 0" in msg
    for key, bad in (("gates", [(t.cs["n_advice"], 0)]), ("gates", [(0, t.cs["n_fixed"])]), ("lookups", [(0, 99)]),
                     ("permutation", [(2, 5)]), ("permutation", [(3, 0)])):
        cs = dict(t.cs, **{key: bad})
        rc, msg = _raw_call(h, cs, *cols)
        assert rc == -1 and "mock_prover" in msg and "out of range" in msg, (key, msg)
    rc, msg = _raw_call(h, dict(t.cs, k=1), *cols)
    assert rc == -1 and "k = 1" in msg


def test_no_device_fails_loudly():
    """without a CUDA device the call fails with H2V_ECUDA: there is no CPU fallback"""
    import halo2_vectordb_b200 as h

    if h.device_count() > 0:
        pytest.skip("GPU present")
    t = Toy(6, seed=2)
    with pytest.raises(h.H2VError, match="no CUDA device"):
        h.MockProver.run(t.cs, *[[fr_arr(c) for c in x] for x in (t.fixed, t.sigma, t.advice, t.instances)])
