"""h2v_create_proofs: many proofs on one key in one call, run in groups phase by phase.

Proof p of a batch must be byte for byte what h2v_create_proof returns for the same advice, instances and seed (and
what the CPU restatement returns), whatever the group size, the number of devices or the streamed-key mode.  The
witnesses of a batch differ (an honest one, three false statements, the honest one under other seeds), so a proof that
read a neighbour's column or challenge would show as a byte difference and as a verifier verdict."""
import copy

import numpy as np
import pytest

from common import fr_arr
from oracle import oracle as O
from oracle import plonk as PL
from toy_circuit import Toy

pytestmark = pytest.mark.gpu

SECRET = 0x1CE1CEBABE5EED0123456789ABCDEF0FEDCBA9876543210


def _seed(i):
    return bytes((i * 37 + j) % 256 for j in range(32))


def _witnesses(t, B):
    """B (toy, seed, honest) triples on t's key: honest, break_gate, break_copy, break_public_input, then the honest
    witness under other seeds"""
    out = []
    for p in range(B):
        w = copy.deepcopy(t)
        how = ("", "break_gate", "break_copy", "break_public_input")[p % 4] if p < 4 else ""
        if how:
            getattr(w, how)()
        out.append((w, _seed(p), not how))
    return out


def _cols(w):
    return [fr_arr(c) for c in w.advice], [fr_arr(c) for c in w.instances]


def _setup(h2v, t, k):
    params = PL.Params.setup(k, SECRET)
    srs = h2v.ParamsKZG(k, params.g, params.g_lagrange)
    pk = h2v.ProvingKey(srs, t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], fr_arr([t.vk_repr])[0])
    return params, srs, pk


def _batch(pk, ws):
    cols = [_cols(w) for w, _, _ in ws]
    return pk.create_proofs([a for a, _ in cols], [i for _, i in cols], [s for _, s, _ in ws])


def _singles(pk, ws):
    return [pk.create_proof(*_cols(w), s) for w, s, _ in ws]


@pytest.mark.parametrize("k,gate_cols,lookup_cols,degree,B",
                         [(6, 2, 1, 4, 1), (6, 3, 2, 4, 2), (7, 1, 1, 5, 3), (6, 4, 0, 4, 5), (8, 5, 3, 4, 8), (6, 2, 1, 6, 3),
                          (10, 6, 2, 4, 2)])
def test_batch_bytes_equal_single_proofs_and_oracle(h2v, k, gate_cols, lookup_cols, degree, B):
    t = Toy(k, seed=k * 100 + gate_cols, n_gate_cols=gate_cols, n_lookup_cols=lookup_cols, degree=degree)
    params, srs, pk = _setup(h2v, t, k)
    ws = _witnesses(t, B)
    got = _batch(pk, ws)
    assert len(got) == B and all(len(g) == pk.proof_size() for g in got)
    assert got == _singles(pk, ws)
    vk = PL.keygen_vk(params, t.cs, t.fixed, t.sigma)
    for g, (w, s, honest) in zip(got, ws):
        assert g == PL.create_proof(params, w.cs, w.fixed, w.sigma, w.vk_repr, w.advice, w.instances, s)
        assert PL.verify_proof(params, w.cs, vk, w.vk_repr, w.instances, g) == honest
    pk.close()
    srs.close()


def test_group_size_changes_no_byte(h2v, monkeypatch):
    k = 8
    t = Toy(k, seed=81, n_gate_cols=4, n_lookup_cols=2)
    params, srs, pk = _setup(h2v, t, k)
    ws = _witnesses(t, 5)
    want = _singles(pk, ws)
    for g in ("1", "2", "3"):
        monkeypatch.setenv("H2V_PROOF_GROUP", g)
        assert _batch(pk, ws) == want, f"H2V_PROOF_GROUP={g}"
    monkeypatch.delenv("H2V_PROOF_GROUP")
    assert _batch(pk, ws) == want
    phases = pk.last_phase_ms()
    assert all(v >= 0 for v in phases.values()) and sum(phases.values()) > 0
    pk.close()
    srs.close()


def test_streamed_key_batch(h2v, monkeypatch):
    """a streamed key (the k = 20 mode, forced at k = 8) proves in groups of one: the same bytes as the resident key's"""
    k = 8
    t = Toy(k, seed=k * 100 + 5, n_gate_cols=5, n_lookup_cols=3)
    params, srs, pk = _setup(h2v, t, k)
    ws = _witnesses(t, 3)
    resident = _singles(pk, ws)
    pk.close()
    monkeypatch.setenv("H2V_STREAM_EXT", "1")
    monkeypatch.setenv("H2V_STREAM_COLS", "6")
    pk = h2v.ProvingKey(srs, t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], fr_arr([t.vk_repr])[0])
    assert _batch(pk, ws) == resident
    pk.close()
    srs.close()


def test_batch_errors_name_the_proof(h2v):
    k = 6
    t = Toy(k, seed=9)
    params, srs, pk = _setup(h2v, t, k)
    ws = _witnesses(t, 4)
    want = _singles(pk, ws)
    bad = copy.deepcopy(ws)
    bad[2][0].advice[t.G][2] = t.tsize + 3                 # proof 2: a lookup value outside the table
    with pytest.raises(ValueError, match="proof 2"):
        _batch(pk, bad)
    assert _batch(pk, ws) == want                          # the key proves correctly afterwards
    cols = [_cols(w) for w, _, _ in ws]
    adv, inst, seeds = [a for a, _ in cols], [i for _, i in cols], [s for _, s, _ in ws]
    with pytest.raises(ValueError, match="proof 1"):       # InstanceTooLarge in proof 1
        pk.create_proofs(adv, inst[:1] + [[fr_arr([1] * (1 << k))]] + inst[2:], seeds)
    with pytest.raises(ValueError, match="proof 3"):       # a short advice list
        pk.create_proofs(adv[:3] + [adv[3][:-1]], inst, seeds)
    with pytest.raises(ValueError):                        # lists of different lengths
        pk.create_proofs(adv, inst[:3], seeds)
    assert pk.create_proofs([], [], []) == []
    # through the C ABI: a stride shorter than a proof, and n_proofs = 0 with nothing else given
    import ctypes as C

    L = h2v.lib()
    size = pk.proof_size()
    out = np.zeros(size, dtype=np.uint8)
    null = C.POINTER(C.c_void_p)()
    assert L.h2v_create_proofs(pk._h, 0, null, null, null, None, None, 0) == 0
    seed = bytes(32)
    a = (C.c_void_p * len(adv[0]))(*[c.ctypes.data for c in adv[0]])
    ia = (C.c_void_p * 1)(*[inst[0][0].ctypes.data])
    il = np.array([inst[0][0].shape[0]], dtype=np.uint32)
    rc = L.h2v_create_proofs(pk._h, 1, (C.c_void_p * 1)(C.cast(a, C.c_void_p)), (C.c_void_p * 1)(C.cast(ia, C.c_void_p)),
                             (C.c_void_p * 1)(il.ctypes.data), seed, out.ctypes.data, size - 1)
    assert rc != 0 and b"stride" in L.h2v_last_error()
    rc = L.h2v_create_proofs(pk._h, 1, (C.c_void_p * 1)(C.cast(a, C.c_void_p)), (C.c_void_p * 1)(C.cast(ia, C.c_void_p)),
                             (C.c_void_p * 1)(il.ctypes.data), seed, out.ctypes.data, size)
    assert rc == 0 and bytes(out) == pk.create_proof(adv[0], inst[0], bytes(32))
    pk.close()
    srs.close()


def _real(Z, name):
    k, bits = Z.EXAMPLE_PARAMS[name]
    inp = Z.example_input(name)
    if name == "query":      # break the five-way ties of data/query.in (tests/test_circuit.py::test_query_layout)
        inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
    return Z.create_circuit(Z.EXAMPLES[name], inp, k, bits)[0]


@pytest.mark.parametrize("name", ["distances", "query"])
def test_batch_of_real_examples(h2v, name):
    from halo2_vectordb_b200 import circuit as Z

    rc = _real(Z, name)
    srs = h2v.ParamsKZG.gen_srs(rc.k)
    pk = h2v.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, np.array([rc.k, 0, 0, 0], dtype=np.uint64))
    seeds = [_seed(p) for p in range(4)]
    got = pk.create_proofs([rc.advice] * 4, [rc.instances] * 4, seeds)
    assert got == [pk.create_proof(rc.advice, rc.instances, s) for s in seeds]
    assert len(set(got)) == 4
    pk.close()
    srs.close()


def test_batch_kmeans_shaped_k16(h2v):
    """k = 16 with a kmeans-like column mix (synthetic_circuit): two proofs in one group, each the single proof, one
    checked against the CPU restatement"""
    from halo2_vectordb_b200.synthetic import synthetic_circuit

    k = 16
    c = synthetic_circuit(k, n_gate_cols=4, n_lookup_cols=2, lookup_bits=15, seed=16)
    s = O.fr_from_ints([SECRET])[0]
    g, gl = h2v.srs_setup(k, s)
    params = PL.Params(k, g, gl, SECRET)
    srs = h2v.ParamsKZG(k, g, gl)
    pk = h2v.ProvingKey(srs, c["cs"], c["fixed"], c["sigma"], c["vk_repr"])
    seeds = [_seed(1), _seed(2)]
    got = pk.create_proofs([c["advice"]] * 2, [c["instances"]] * 2, seeds)
    assert got == [pk.create_proof(c["advice"], c["instances"], s_) for s_ in seeds]
    ints = lambda cols: [O.fr_to_ints(col) for col in cols]
    vk_repr = O.fr_to_ints(c["vk_repr"].reshape(1, 4))[0]
    assert got[1] == PL.create_proof(params, c["cs"], ints(c["fixed"]), ints(c["sigma"]), vk_repr, ints(c["advice"]),
                                     ints(c["instances"]), seeds[1])
    pk.close()
    srs.close()


def test_batch_on_two_devices(h2v):
    """h2v_init([0, 1]): the larger batches split over the devices; the bytes do not depend on the device count"""
    if h2v.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    k = 9
    t = Toy(k, seed=93, n_gate_cols=6, n_lookup_cols=2)
    ws = _witnesses(t, 6)
    _, srs, pk = _setup(h2v, t, k)
    one = _batch(pk, ws)
    pk.close()
    srs.close()
    h2v.init([0, 1])
    try:
        _, srs, pk = _setup(h2v, t, k)
        assert _batch(pk, ws) == one
        pk.close()
        srs.close()
    finally:
        h2v.init(0)
