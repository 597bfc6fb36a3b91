"""h2v_pk_mock_prover: the mock prover on a loaded proving key, for a batch of witnesses in one call.

Witness w's failures and total must be exactly what h2v_mock_prover returns for the key's constraint system, fixed and
sigma columns and witness w's advice and instances, whatever the group size, the call (first or later), the key mode or
the device count; and a check must change no proof.  h2v_mock_prover runs the same key-table and check code (a batch of
one), so comparing with it shows that batching, grouping and the key's resident columns change nothing, not that the
checks are right.  The independent references are oracle/mock.py, whose messages the toy and malformed-key cases are
compared with (as tests/test_mock_prover.py does for h2v_mock_prover), and the known totals of the real layouts
(data/query.in's 12 gate failures, kmeans' 0)."""
import copy
import ctypes as C

import numpy as np
import pytest

from common import fr_arr
from oracle import mock as M
from oracle import oracle as O
from oracle import pyref as P
from test_mock_prover import BIG, TOYS, _messages
from toy_circuit import Toy

R = P.R
SECRET = 0x1CE1CEBABE5EED0123456789ABCDEF0FEDCBA9876543210


# ----------------------------------------------------------------------------------------------- helpers
def _srs(h, k):
    g, gl = h.srs_setup(k, O.fr_from_ints([SECRET])[0])
    srs = h.ParamsKZG(k, g, gl)
    srs.g, srs.g_lagrange = g, gl
    return srs


def _key(h, t, srs=None):
    srs = srs or _srs(h, t.k)
    return srs, h.ProvingKey(srs, t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], fr_arr([t.vk_repr])[0])


def _cols(w):
    return [fr_arr(c) for c in w.advice], [fr_arr(c) for c in w.instances]


def _witnesses(t):
    """honest, break_gate, break_copy, break_public_input, a lookup input moved out of its table, honest"""
    out = []
    for how in ("", "break_gate", "break_copy", "break_public_input", "lookup", ""):
        w = copy.deepcopy(t)
        if how == "lookup":
            if t.Lc:
                w.advice[t.G][2] = t.tsize + 3
        elif how:
            getattr(w, how)()
        out.append(w)
    return out


def _check_batch(h, pk, cs, fixed, sigma, batch, cap=4096):
    """pk.mock_prover on the batch [(advice, instances)] equals MockProver.run on each witness's columns"""
    got = pk.mock_prover([a for a, _ in batch], [i for _, i in batch], max_failures=cap)
    assert len(got) == len(batch)
    for w, ((adv, inst), mp) in enumerate(zip(batch, got)):
        want = h.MockProver.run(cs, fixed, sigma, adv, inst, max_failures=cap)
        assert (mp.failures, mp.n_failures) == (want.failures, want.n_failures), f"witness {w}"
    return got


def _toy_batch(h, t, pk, ws, cap=4096):
    return _check_batch(h, pk, t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], [_cols(w) for w in ws], cap)


# ----------------------------------------------------------------------------------------------- toy keys
@pytest.mark.gpu
@pytest.mark.parametrize("k,seed,gate_cols,lookup_cols,degree", [t + (4,) for t in TOYS] + [(7, 11, 2, 2, 5), (8, 12, 3, 1, 6)])
def test_toy_batch_equals_single_checks_and_oracle(h2v, k, seed, gate_cols, lookup_cols, degree):
    t = Toy(k, seed=seed, n_gate_cols=gate_cols, n_lookup_cols=lookup_cols, degree=degree)
    srs, pk = _key(h2v, t)
    ws = _witnesses(t)
    got = _toy_batch(h2v, t, pk, ws)
    for w, mp in zip(ws, got):
        want = M.mock_prover(t.cs, t.fixed, t.sigma, w.advice, w.instances, max_failures=BIG)
        assert _messages(h2v, t.cs, mp.failures, t.fixed, w.advice, w.instances) == want
        assert mp.n_failures == len(want)
    assert got[0].n_failures == 0 and got[-1].n_failures == 0
    assert got[1].n_failures and got[2].n_failures      # break_gate, break_copy
    for mp in got:
        if mp.n_failures:
            with pytest.raises(AssertionError, match="not satisfied"):
                mp.assert_satisfied()
        else:
            mp.assert_satisfied()
    if lookup_cols:
        assert any(f.kind == h2v.MOCK_LOOKUP for f in got[4].failures)
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_caps(h2v):
    t = Toy(8, seed=21, n_gate_cols=3, n_lookup_cols=2)
    srs, pk = _key(h2v, t)
    ws = _witnesses(t)
    full = _toy_batch(h2v, t, pk, ws)
    total = max(mp.n_failures for mp in full)
    assert total >= 2
    for cap in (0, 1, total - 1):
        got = _toy_batch(h2v, t, pk, ws, cap=cap)
        for a, b in zip(got, full):
            assert a.failures == b.failures[:cap] and a.n_failures == b.n_failures
    assert pk.mock_prover([], []) == []
    assert h2v.lib().h2v_pk_mock_prover(pk._h, 0, None, None, None, None, 0, None) == 0
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_key_state(h2v, monkeypatch):
    """later calls and forced group sizes give the first call's output; a check changes no proof"""
    k = 8
    t = Toy(k, seed=31, n_gate_cols=4, n_lookup_cols=2)
    srs, pk = _key(h2v, t)
    ws = _witnesses(t)
    adv, inst = _cols(ws[0])
    seed = bytes(range(32))
    first = _toy_batch(h2v, t, pk, ws)
    assert [(m.failures, m.n_failures) for m in _toy_batch(h2v, t, pk, ws)] == [(m.failures, m.n_failures) for m in first]
    for g in ("1", "2"):
        monkeypatch.setenv("H2V_PROOF_GROUP", g)
        got = _toy_batch(h2v, t, pk, ws)
        assert [(m.failures, m.n_failures) for m in got] == [(m.failures, m.n_failures) for m in first], g
    monkeypatch.delenv("H2V_PROOF_GROUP")
    checked = pk.create_proof(adv, inst, seed)
    batch = pk.create_proofs([_cols(w)[0] for w in ws[:2]], [_cols(w)[1] for w in ws[:2]], [seed, seed])
    pk.close()
    _, fresh = _key(h2v, t, srs)
    assert checked == fresh.create_proof(adv, inst, seed)
    assert batch == fresh.create_proofs([_cols(w)[0] for w in ws[:2]], [_cols(w)[1] for w in ws[:2]], [seed, seed])
    fresh.close()
    srs.close()


@pytest.mark.gpu
def test_malformed_key(h2v):
    """a sigma cell that is not delta^c omega^r and two cells with one image: every witness reports them as
    h2v_mock_prover does"""
    t = Toy(8, seed=17, n_gate_cols=3, n_lookup_cols=2)
    pc = t.cs["permutation"].index((0, 0))
    t.sigma[pc + 1][5] = 12345
    t.sigma[pc][9] = t.sigma[pc][10]
    srs, pk = _key(h2v, t)
    ws = _witnesses(t)
    got = _toy_batch(h2v, t, pk, ws)
    key_kinds = {h2v.MOCK_SIGMA_NOT_DELTA_OMEGA, h2v.MOCK_SIGMA_NOT_PERMUTATION}
    key_only = [f for f in got[0].failures if f.kind in key_kinds]
    assert {f.kind for f in key_only} == key_kinds
    for w, mp in zip(ws, got):
        assert [f for f in mp.failures if f.kind in key_kinds] == key_only
        want = M.mock_prover(t.cs, t.fixed, t.sigma, w.advice, w.instances, max_failures=BIG)
        assert _messages(h2v, t.cs, mp.failures, t.fixed, w.advice, w.instances) == want
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_unreduced_limbs(h2v):
    """advice and instance values given as value + r are the same field elements: no failure"""
    t = Toy(7, seed=3, n_gate_cols=2, n_lookup_cols=1)
    srs, pk = _key(h2v, t)

    def unreduce(col):
        raw = O.limbs_to_ints(col)
        return O.ints_to_limbs([x + R if x + R < 1 << 256 else x for x in raw])

    adv, inst = _cols(t)
    adv2, inst2 = [unreduce(c) for c in adv], [unreduce(c) for c in inst]
    assert sum(int((a != b).any(axis=1).sum()) for a, b in zip(adv, adv2)) > t.n
    got = pk.mock_prover([adv, adv2], [inst, inst2])
    assert [(m.failures, m.n_failures) for m in got] == [([], 0), ([], 0)]
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_streamed_key(h2v, monkeypatch):
    k = 8
    t = Toy(k, seed=41, n_gate_cols=5, n_lookup_cols=3)
    ws = _witnesses(t)
    srs, pk = _key(h2v, t)
    resident = [(m.failures, m.n_failures) for m in _toy_batch(h2v, t, pk, ws)]
    pk.close()
    monkeypatch.setenv("H2V_STREAM_EXT", "1")
    monkeypatch.setenv("H2V_STREAM_COLS", "6")
    _, pk = _key(h2v, t, srs)
    assert [(m.failures, m.n_failures) for m in _toy_batch(h2v, t, pk, ws)] == resident
    pk.close()
    srs.close()


# ----------------------------------------------------------------------------------------------- the examples
def _layout(Z, name, inp=None):
    k0, lb0 = Z.EXAMPLE_PARAMS[name]
    return Z.create_circuit(Z.EXAMPLES[name], inp or Z.example_input(name), k0, lb0)[0]


def _real_key(h, rc):
    srs = _srs(h, rc.k)
    return srs, h.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, np.array([rc.k, 0, 0, 0], dtype=np.uint64))


@pytest.mark.gpu
def test_distances_and_query(h2v):
    from halo2_vectordb_b200 import circuit as Z

    rc = _layout(Z, "distances")
    srs, pk = _real_key(h2v, rc)
    bad = list(rc.advice)
    bad[0] = bad[0].copy()
    bad[0][7] = fr_arr([O.fr_to_ints(np.ascontiguousarray(bad[0][7:8]))[0] + 1])[0]
    got = _check_batch(h2v, pk, rc.cs, rc.fixed, rc.sigma, [(rc.advice, rc.instances), (bad, rc.instances), (rc.advice, rc.instances)])
    assert got[0].n_failures == 0 and got[1].n_failures >= 2 and got[2].n_failures == 0
    pk.close()
    srs.close()
    rc = _layout(Z, "query")
    srs, pk = _real_key(h2v, rc)
    got = _check_batch(h2v, pk, rc.cs, rc.fixed, rc.sigma, [(rc.advice, rc.instances)] * 3)
    for mp in got:      # data/query.in's five-way ties: 12 gate failures
        assert mp.n_failures == 12 and all(f.kind == h2v.MOCK_GATE for f in mp.failures)
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_kmeans_honest_batch(h2v):
    from halo2_vectordb_b200 import circuit as Z

    rc = _layout(Z, "kmeans")
    srs, pk = _real_key(h2v, rc)
    got = pk.mock_prover([rc.advice] * 2, [rc.instances] * 2)
    assert [(m.failures, m.n_failures) for m in got] == [([], 0), ([], 0)]
    pk.close()
    srs.close()


# ----------------------------------------------------------------------------------------------- errors
def _raw(h, pk, advs, insts, lens, cap=4):
    B = len(advs)
    keep = []

    def lst(cols):
        a = (C.c_void_p * max(1, len(cols)))(*[None if c is None else c.ctypes.data for c in cols])
        keep.append(a)
        return C.cast(a, C.c_void_p)

    ap = (C.c_void_p * B)(*[lst(a) for a in advs])
    ip = (C.c_void_p * B)(*[lst(i) for i in insts])
    ls = [np.ascontiguousarray(x, dtype=np.uint32) for x in lens]
    lp = (C.c_void_p * B)(*[x.ctypes.data for x in ls])
    out = (h._MockFailureT * max(1, B * cap))()
    totals = np.zeros(B, dtype=np.uint64)
    rc = h.lib().h2v_pk_mock_prover(pk._h, B, ap, ip, lp, out, cap, totals.ctypes.data)
    return rc, h.lib().h2v_last_error().decode()


@pytest.mark.gpu
def test_errors_name_the_witness_and_leave_the_key_usable(h2v):
    k = 6
    t = Toy(k, seed=9)
    srs, pk = _key(h2v, t)
    seed = bytes(32)
    adv, inst = _cols(t)
    want = pk.create_proof(adv, inst, seed)
    lens = [c.shape[0] for c in inst]
    advs, insts = [adv] * 4, [inst] * 4
    launches = h2v.launch_count()
    rc, msg = _raw(h2v, pk, advs, insts, [lens, lens, [t.n + 1], lens])
    assert rc == -1 and "witness 2" in msg and "instance column 0" in msg, msg
    rc, msg = _raw(h2v, pk, advs[:1] + [adv[:1] + [None] + adv[2:]] + advs[2:], insts, [lens] * 4)
    assert rc == -1 and "witness 1" in msg and "advice column 1 is NULL" in msg, msg
    rc, msg = _raw(h2v, pk, advs, insts[:3] + [[None]], [lens] * 4)
    assert rc == -1 and "witness 3" in msg and "instance column 0 is NULL" in msg, msg
    assert h2v.launch_count() == launches          # rejected before any device work
    L = h2v.lib()
    assert L.h2v_pk_mock_prover(None, 1, None, None, None, None, 0, None) == -1 and b"NULL key" in L.h2v_last_error()
    totals = np.zeros(1, dtype=np.uint64)
    assert L.h2v_pk_mock_prover(pk._h, 1, None, None, None, None, 0, totals.ctypes.data) == -1
    assert b"NULL argument" in L.h2v_last_error()
    with pytest.raises(ValueError, match="witness 1"):
        pk.mock_prover([adv, adv[:-1]], [inst, inst])
    with pytest.raises(ValueError):
        pk.mock_prover([adv], [inst, inst])
    assert pk.mock_prover([adv], [inst])[0].n_failures == 0
    assert pk.create_proof(adv, inst, seed) == want          # the key proves correctly afterwards
    pk.close()
    srs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("limit", ["gates", "flags"])
def test_limits(h2v, limit):
    """keys h2v_pk_load accepts but the checks cannot take: more than 65535 gates (every gate on the same columns), or
    2^32 flags per witness (k = 16, 65535 gates and one lookup)"""
    k, G, L = (4, 65536, 0) if limit == "gates" else (16, 65535, 1)
    n = 1 << k
    cs = dict(k=k, degree=4, blinding_factors=1, n_advice=1, n_fixed=1, n_instance=0, gates=[(0, 0)] * G,
              lookups=[(0, 0)] * L, permutation=[], advice_queries=[(0, 0)], fixed_queries=[(0, 0)])
    zero = np.zeros((n, 4), dtype=np.uint64)
    srs = _srs(h2v, k)
    pk = h2v.ProvingKey(srs, cs, [zero], [], np.zeros(4, dtype=np.uint64))
    with pytest.raises(ValueError, match="pk_mock_prover: " + ("more than 65535 gates" if limit == "gates" else r".*more than 2\^32")):
        pk.mock_prover([[zero]], [[]])
    pk.close()
    srs.close()


@pytest.mark.gpu
def test_two_devices(h2v):
    if h2v.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    t = Toy(8, seed=51, n_gate_cols=4, n_lookup_cols=2)
    ws = _witnesses(t)
    results = []
    for devs in ([0], [0, 1]):
        h2v.init(devs)
        srs, pk = _key(h2v, t)
        results.append([(m.failures, m.n_failures) for m in _toy_batch(h2v, t, pk, ws)])
        pk.close()
        srs.close()
    h2v.init(0)
    assert results[0] == results[1]


# ----------------------------------------------------------------------------------------------- no device needed
def test_symbol_exported_and_declared():
    import os
    import re

    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import build

    build.build()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "h2v.h")).read()
    assert re.search(r"\bint h2v_pk_mock_prover\s*\(", hdr)
    assert "h2v_pk_mock_prover" in h.ABI_SYMBOLS
    assert hasattr(h.lib(), "h2v_pk_mock_prover")
    assert "h2v_pk_mock_prover" in open(os.path.join(root, "include", "h2v.hpp")).read()


def test_no_device_fails_loudly():
    """Without a CUDA device there is no key to check against: loading one fails with H2V_ECUDA (no CPU fallback), as
    h2v_mock_prover does, and h2v_pk_mock_prover on a NULL key is refused with H2V_EINVAL.  It cannot be called on a key
    without a device, so H2V_ECUDA from the call itself is not reachable here."""
    import halo2_vectordb_b200 as h

    if h.device_count() > 0:
        pytest.skip("GPU present")
    t = Toy(6, seed=2)
    with pytest.raises(h.H2VError, match="no CUDA device"):
        h.MockProver.run(t.cs, *[[fr_arr(c) for c in x] for x in (t.fixed, t.sigma, t.advice, t.instances)])
    with pytest.raises(h.H2VError):
        _key(h, t)
    assert h.lib().h2v_pk_mock_prover(None, 1, None, None, None, None, 0, None) == -1


# ----------------------------------------------------------------------------------------------- the C++ mirror
def _compile_cpp(tmp_path):
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "cpp_pk_mock_check")
    libdir = os.path.join(root, "halo2_vectordb_b200")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I" + os.path.join(root, "include"), "-o", exe,
                           os.path.join(root, "tests", "cpp_pk_mock_check.cpp"), "-L" + libdir, "-lh2v", "-Wl,-rpath," + libdir])
    return exe


def _write_case(path, t, srs, ws, cap):
    """the input of tests/cpp_pk_mock_check.cpp: t's circuit, key columns and SRS, and the witnesses ws"""
    cs = t.cs
    u32 = lambda xs: np.asarray(xs, dtype=np.uint32).tobytes()
    parts = [u32([cs["k"], cs["degree"], cs["blinding_factors"], cs["n_advice"], cs["n_fixed"], cs["n_instance"], len(cs["gates"]),
                  len(cs["lookups"]), len(cs["permutation"]), len(cs["advice_queries"]), len(cs["fixed_queries"]), len(ws), cap]),
             u32([g[0] for g in cs["gates"]]), u32([g[1] for g in cs["gates"]]),
             u32([l[0] for l in cs["lookups"]]), u32([l[1] for l in cs["lookups"]]),
             np.asarray([p[0] for p in cs["permutation"]], dtype=np.uint8).tobytes(), u32([p[1] for p in cs["permutation"]]),
             u32([q[0] for q in cs["advice_queries"]]), np.asarray([q[1] for q in cs["advice_queries"]], dtype=np.int32).tobytes(),
             u32([q[0] for q in cs["fixed_queries"]]), np.asarray([q[1] for q in cs["fixed_queries"]], dtype=np.int32).tobytes(),
             np.ascontiguousarray(srs.g).tobytes(), np.ascontiguousarray(srs.g_lagrange).tobytes()]
    parts += [fr_arr(c).tobytes() for c in t.fixed] + [fr_arr(c).tobytes() for c in t.sigma] + [fr_arr([t.vk_repr]).tobytes()]
    for w in ws:
        adv, inst = _cols(w)
        parts += [a.tobytes() for a in adv]
        for c in inst:
            parts += [u32([c.shape[0]]), c.tobytes()]
    with open(path, "wb") as f:
        f.write(b"".join(parts))


def test_cpp_mirror_compiles_and_fails_loudly_without_gpu(tmp_path):
    import subprocess

    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import build

    build.build()
    exe = _compile_cpp(tmp_path)
    if h.device_count() == 0:
        out = subprocess.run([exe], capture_output=True, text=True)
        assert out.returncode == 0 and "no device" in out.stdout, out.stdout + out.stderr


@pytest.mark.gpu
def test_cpp_mirror_batch(h2v, tmp_path):
    """h2v_host::ProvingKey::mock_prover gives Python's ProvingKey.mock_prover output for every witness"""
    import subprocess

    t = Toy(8, seed=61, n_gate_cols=3, n_lookup_cols=2)
    ws = _witnesses(t)
    srs, pk = _key(h2v, t)
    want = _toy_batch(h2v, t, pk, ws, cap=16)
    case = str(tmp_path / "case.bin")
    _write_case(case, t, srs, ws, 16)
    out = subprocess.run([_compile_cpp(tmp_path), case], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    got, lines = [], out.stdout.splitlines()
    for line in lines:
        f = line.split()
        if f[0] == "witness":
            got.append(([], int(f[2])))
        else:
            got[-1][0].append(h2v.MockFailure(*map(int, f)))
    assert got == [(m.failures, m.n_failures) for m in want]
    assert any(n for _, n in got)
    pk.close()
    srs.close()
