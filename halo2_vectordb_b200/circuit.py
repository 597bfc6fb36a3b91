"""Host-side mirror of the reference's chip API over the C ABI's circuit builder (SURVEY.md 8(f) row 4).

Same names, argument meaning and failure behaviour as the reference, so that tests read like the reference's own
(/root/reference/tests/distances/mod.rs, tests/vectordb/mod.rs) and the three example circuits
(/root/reference/examples/{distances,query,kmeans}.rs) can be restated line by line:

    builder = GateThreadBuilder(lookup_bits=12)          # halo2-base GateThreadBuilder + LOOKUP_BITS
    ctx = builder.main(0)
    fp = FixedPointChip.default(builder)                 # FixedPointChip::<F, 48>::default(lookup_bits)
    dist = DistanceChip.default(fp)
    a = ctx.assign_witnesses(fp.quantize_vector([0.1, 0.2]))
    d = dist.euclidean_distance(ctx, a, b);  fp.dequantization(d.value())

All the work happens in libh2v.so (csrc/zk_builder.hpp, zk_chips.hpp, circuit.cu); this file only marshals cell indices.
`RangeCircuit` lays the trace out into the columns `ProvingKey` / `create_proof` take.  `WitnessProgram` replays a recorded
circuit for many new inputs on the GPU and gives the same advice columns and instances without the host builder.
"""
import ctypes as C

import numpy as np

from . import BUILDER_SYMBOLS, H2VError, _check, _fr, _fr1, _ptr, lib

(FP_QADD, FP_QSUB, FP_QMUL, FP_QDIV, FP_QMOD, FP_QPOW, FP_QMAX, FP_QMIN, FP_BIT_XOR, FP_COND_NEG) = range(1, 11)
(FP_NEG, FP_QABS, FP_IS_NEG, FP_SIGN, FP_CLIP, FP_QEXP2, FP_QLOG2, FP_QEXP, FP_QLOG, FP_QSQRT, FP_QSIN, FP_QCOS, FP_QTAN,
 FP_QSINH, FP_QCOSH, FP_QTANH) = range(20, 36)
FP_QSUM, FP_INNER_PRODUCT, FP_POLYNOMIAL = 40, 41, 42
DISTANCE_EUCLIDEAN, DISTANCE_COSINE, DISTANCE_HAMMING, DISTANCE_MANHATTAN = 60, 61, 62, 63


_i64p = C.POINTER(C.c_int64)
_u64pp = C.POINTER(C.POINTER(C.c_uint64))
_typed = False


def _L():
    global _typed
    L = lib()
    if not _typed:
        L.h2v_builder_new.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        L.h2v_builder_free.argtypes = [C.c_void_p]
        L.h2v_builder_free.restype = None
        L.h2v_builder_quantize.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_dequantize.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_assign_witnesses.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_load_constant.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_builder_cell_values.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_make_public.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        L.h2v_builder_call.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_nearest_vector.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p]
        L.h2v_builder_kmeans.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_size_t, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        L.h2v_builder_poseidon_new.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
        L.h2v_builder_poseidon_hash.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.h2v_builder_merkle_commitment.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]
        L.h2v_builder_stats.argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_builder_config.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
        L.h2v_builder_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_builder_layout.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        L.h2v_layout_free.argtypes = [C.c_void_p]
        L.h2v_layout_free.restype = None
        L.h2v_layout_info.argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_layout_columns.argtypes = [C.c_void_p, C.c_int, C.POINTER(_u64pp), C.POINTER(C.c_size_t)]
        L.h2v_layout_instance.argtypes = [C.c_void_p, C.POINTER(C.POINTER(C.c_uint64)), C.POINTER(C.c_size_t)]
        L.h2v_layout_break_points.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.h2v_builder_new_recording.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        L.h2v_witness_program_new.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
        L.h2v_witness_program_free.argtypes = [C.c_void_p]
        L.h2v_witness_program_free.restype = None
        L.h2v_witness_program_info.argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_witness_program_inputs.argtypes = [C.c_void_p, C.c_void_p]
        L.h2v_witness_program_rule_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.h2v_witness_generate.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
        L.h2v_witness_last_ms.argtypes = [C.POINTER(C.c_double)]
        _typed = True
    return L


class AssignedValue:
    """halo2-base `AssignedValue<F>`: a cell of the execution trace."""
    __slots__ = ("builder", "cell")

    def __init__(self, builder, cell):
        self.builder, self.cell = builder, int(cell)

    def value(self):
        """the cell's value (Montgomery-form limbs, like every Fr that crosses the C ABI)"""
        return self.builder.cell_values([self])[0]

    def __repr__(self):
        return f"AssignedValue(cell={self.cell})"


def _cells(vs):
    return np.ascontiguousarray([v.cell for v in vs], dtype=np.int64)


class Context:
    """halo2-base `Context<F>` (the single thread `builder.main(0)`, /root/reference/src/scaffold/mod.rs:61)"""

    def __init__(self, builder):
        self.builder = builder

    def assign_witnesses(self, values):
        vals = _fr(np.asarray(values, dtype=np.uint64).reshape(-1, 4))
        out = np.zeros(vals.shape[0], dtype=np.int64)
        _check(_L().h2v_builder_assign_witnesses(self.builder._h, _ptr(vals), vals.shape[0], _ptr(out)))
        return [AssignedValue(self.builder, c) for c in out]

    def load_witness(self, value):
        return self.assign_witnesses([value])[0]

    def load_constant(self, value):
        out = C.c_int64()
        _check(_L().h2v_builder_load_constant(self.builder._h, _ptr(_fr1(value)), C.byref(out)))
        return AssignedValue(self.builder, out.value)


class GateThreadBuilder:
    """halo2-base `GateThreadBuilder<Fr>` together with the `LOOKUP_BITS` the scaffold reads from the environment
    (mod.rs:361-372) and the PRECISION_BITS of the chips built over it (48 in every example).  record=True also keeps
    the rule of every cell, so that `WitnessProgram` can replay the circuit for other inputs."""

    def __init__(self, lookup_bits, precision_bits=48, record=False):
        self.lookup_bits, self.precision_bits, self.record = lookup_bits, precision_bits, record
        self._h = C.c_void_p()
        new = _L().h2v_builder_new_recording if record else _L().h2v_builder_new
        _check(new(precision_bits, lookup_bits, C.byref(self._h)))
        self._ctx = Context(self)
        self.assigned_instances = []

    @classmethod
    def mock(cls, lookup_bits, precision_bits=48):
        return cls(lookup_bits, precision_bits)

    def main(self, phase=0):
        if phase != 0:
            raise ValueError("only phase 0 exists in the reference's circuits")
        return self._ctx

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _L().h2v_builder_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def cell_values(self, cells):
        idx = _cells(cells)
        out = np.zeros((len(idx), 4), dtype=np.uint64)
        _check(_L().h2v_builder_cell_values(self._h, _ptr(idx), len(idx), _ptr(out)))
        return out

    def make_public(self, cells):
        """the scaffold's `make_public: &mut Vec<AssignedValue<F>>` (mod.rs:376)"""
        idx = _cells(cells)
        _check(_L().h2v_builder_make_public(self._h, _ptr(idx), len(idx)))
        self.assigned_instances.extend(cells)

    def call(self, op, cells):
        idx = _cells(cells)
        out = C.c_int64()
        _check(_L().h2v_builder_call(self._h, op, _ptr(idx), len(idx), C.byref(out)))
        return AssignedValue(self, out.value)

    def stats(self):
        out = np.zeros(4, dtype=np.uint64)
        _check(_L().h2v_builder_stats(self._h, _ptr(out)))
        return dict(advice_cells=int(out[0]), lookup_cells=int(out[1]), constants=int(out[2]), instances=int(out[3]))

    def config(self, k, minimum_rows=9):
        """`builder.config(k, Some(minimum_rows))` (mod.rs:383-388) -> FlexGateConfigParams"""
        out = np.zeros(3, dtype=np.uint32)
        _check(_L().h2v_builder_config(self._h, k, minimum_rows, _ptr(out)))
        return dict(strategy="Vertical", k=k, num_advice_per_phase=[int(out[0])], num_lookup_advice_per_phase=[int(out[1])],
                    num_fixed=int(out[2]))

    def trace(self):
        """(advice cells as canonical limbs, gate selectors, offsets of the lookup cells)"""
        st = self.stats()
        adv = np.zeros((st["advice_cells"], 4), dtype=np.uint64)
        sel = np.zeros(st["advice_cells"], dtype=np.uint8)
        lk = np.zeros(st["lookup_cells"], dtype=np.int64)
        _check(_L().h2v_builder_trace(self._h, _ptr(adv), _ptr(sel), _ptr(lk)))
        return adv, sel, lk


class FixedPointChip:
    """/root/reference/src/gadget/fixed_point.rs `FixedPointChip<F, PRECISION_BITS>` + `FixedPointInstructions`"""

    def __init__(self, builder):
        self.builder = builder
        self.lookup_bits, self.precision_bits = builder.lookup_bits, builder.precision_bits

    @classmethod
    def default(cls, builder):
        return cls(builder)

    # fixed_point.rs:104-136, fixed_point_vec.rs
    def quantization(self, x):
        return self.quantize_vector([x])[0]

    def quantize_vector(self, v):
        x = np.ascontiguousarray(v, dtype=np.float64)
        out = np.zeros((x.size, 4), dtype=np.uint64)
        _check(_L().h2v_builder_quantize(self.builder._h, _ptr(x), x.size, _ptr(out)))
        return out

    def dequantization(self, x):
        return self._deq(np.asarray(x, dtype=np.uint64).reshape(1, 4))[0]

    def _deq(self, arr):
        arr = _fr(arr)
        out = np.zeros(arr.shape[0], dtype=np.float64)
        _check(_L().h2v_builder_dequantize(self.builder._h, _ptr(arr), arr.shape[0], _ptr(out)))
        return [float(v) for v in out]

    def dequantize_vector(self, cells):
        return self._deq(self.builder.cell_values(cells))

    def quantize_and_assign_vector(self, ctx, v):
        return ctx.assign_witnesses(self.quantize_vector(v))


def _binary(op):
    def f(self, ctx, a, b):
        return self.builder.call(op, [a, b])
    return f


def _unary(op):
    def f(self, ctx, a):
        return self.builder.call(op, [a])
    return f


for _name, _op in dict(qadd=FP_QADD, qsub=FP_QSUB, qmul=FP_QMUL, qdiv=FP_QDIV, qmod=FP_QMOD, qpow=FP_QPOW, qmax=FP_QMAX, qmin=FP_QMIN,
                       bit_xor=FP_BIT_XOR, cond_neg=FP_COND_NEG).items():
    setattr(FixedPointChip, _name, _binary(_op))
for _name, _op in dict(neg=FP_NEG, qabs=FP_QABS, is_neg=FP_IS_NEG, sign=FP_SIGN, clip=FP_CLIP, qexp2=FP_QEXP2, qlog2=FP_QLOG2, qexp=FP_QEXP,
                       qlog=FP_QLOG, qsqrt=FP_QSQRT, qsin=FP_QSIN, qcos=FP_QCOS, qtan=FP_QTAN, qsinh=FP_QSINH, qcosh=FP_QCOSH,
                       qtanh=FP_QTANH).items():
    setattr(FixedPointChip, _name, _unary(_op))
FixedPointChip.qsum = lambda self, ctx, a: self.builder.call(FP_QSUM, list(a))
FixedPointChip.inner_product = lambda self, ctx, a, b: self.builder.call(FP_INNER_PRODUCT, list(a) + list(b))
FixedPointChip.polynomial = lambda self, ctx, x, coef: self.builder.call(FP_POLYNOMIAL, [x] + list(coef))


class DistanceChip:
    """/root/reference/src/gadget/distance.rs `DistanceChip` + `DistanceInstructions`"""

    def __init__(self, fixed_point_gate):
        self.fixed_point_gate = fixed_point_gate
        self.builder = fixed_point_gate.builder

    @classmethod
    def default(cls, fixed_point_gate):
        return cls(fixed_point_gate)

    def _d(self, op, a, b):
        if len(a) != len(b):
            raise ValueError("assertion failed: a.len() == b.len()")      # distance.rs:106,130,155,186
        return self.builder.call(op, list(a) + list(b))

    def euclidean_distance(self, ctx, a, b):
        return self._d(DISTANCE_EUCLIDEAN, a, b)

    def cosine_distance(self, ctx, a, b):
        return self._d(DISTANCE_COSINE, a, b)

    def hamming_distance(self, ctx, a, b):
        return self._d(DISTANCE_HAMMING, a, b)

    def manhattan_distance(self, ctx, a, b):
        return self._d(DISTANCE_MANHATTAN, a, b)


class PoseidonChip:
    """halo2-base `PoseidonChip<F, T, RATE>` (examples/query.rs:27-30, 68): clear / update / squeeze"""

    def __init__(self, ctx, r_f, r_p, t=3, rate=2):
        self.builder = ctx.builder
        _check(_L().h2v_builder_poseidon_new(self.builder._h, t, rate, r_f, r_p))
        self._buf = []

    def clear(self):
        self._buf = []

    def update(self, cells):
        self._buf.extend(cells)

    def squeeze(self, ctx, gate=None):
        idx = _cells(self._buf)
        self._buf = []
        out = C.c_int64()
        _check(_L().h2v_builder_poseidon_hash(self.builder._h, _ptr(idx), len(idx), C.byref(out)))
        return AssignedValue(self.builder, out.value)


class VectorDBChip:
    """/root/reference/src/gadget/vectordb.rs `VectorDBChip` + `VectorDBInstructions`; `distance` is one of the
    DISTANCE_* constants (the reference passes a closure over DistanceChip; the four choices are the chip's methods)"""

    def __init__(self, fixed_point_gate):
        self.fixed_point_gate = fixed_point_gate
        self.builder = fixed_point_gate.builder

    @classmethod
    def default(cls, fixed_point_gate):
        return cls(fixed_point_gate)

    @staticmethod
    def _matrix(vectors):
        dim = len(vectors[0]) if vectors else 0
        if any(len(v) != dim for v in vectors):
            raise ValueError("vectors must have equal lengths")
        return np.ascontiguousarray([[c.cell for c in v] for v in vectors], dtype=np.int64).reshape(len(vectors), dim), dim

    def nearest_vector(self, ctx, query, vectors, distance):
        m, dim = self._matrix(vectors)
        if len(query) != dim:
            raise ValueError("assertion failed: a.len() == b.len()")
        ind = np.zeros(len(vectors), dtype=np.int64)
        res = np.zeros(dim, dtype=np.int64)
        _check(_L().h2v_builder_nearest_vector(self.builder._h, distance, _ptr(_cells(query)), _ptr(m), len(vectors), dim, _ptr(ind), _ptr(res)))
        return [AssignedValue(self.builder, c) for c in ind], [AssignedValue(self.builder, c) for c in res]

    def merkle_commitment(self, ctx, poseidon, vectors):
        m, dim = self._matrix(vectors)
        out = C.c_int64()
        _check(_L().h2v_builder_merkle_commitment(self.builder._h, _ptr(m), len(vectors), dim, C.byref(out)))
        return AssignedValue(self.builder, out.value)

    def kmeans(self, ctx, vectors, distance, K, I):
        m, dim = self._matrix(vectors)
        cen = np.zeros((K, dim), dtype=np.int64)
        ind = np.zeros((len(vectors), K), dtype=np.int64)
        _check(_L().h2v_builder_kmeans(self.builder._h, distance, _ptr(m), len(vectors), dim, K, I, _ptr(cen), _ptr(ind)))
        wrap = lambda a: [[AssignedValue(self.builder, c) for c in row] for row in a]
        return wrap(cen), wrap(ind)


class RangeCircuit:
    """`RangeWithInstanceCircuitBuilder` over `RangeCircuitBuilder::{mock, keygen, prover}(builder)`
    (/root/reference/src/scaffold/mod.rs:391-400): the laid-out columns plus the constraint-system description
    `ProvingKey` takes.  Column views point into the layout and stay valid while this object lives."""

    BLINDING_FACTORS = 6      # max(3, 4 rotations of the vertical gate) + 2; the scaffold's MINIMUM_ROWS = 9 = 6 + 3

    def __init__(self, builder, k, minimum_rows=9):
        self.builder = builder
        self._h = C.c_void_p()
        _check(_L().h2v_builder_layout(builder._h, k, minimum_rows, C.byref(self._h)))
        info = np.zeros(8, dtype=np.uint32)
        _check(_L().h2v_layout_info(self._h, _ptr(info)))
        self.k, self.num_advice, self.num_lookup_advice, self.num_fixed, self.num_instances = (int(x) for x in info[:5])
        self.lookup_bits = int(info[6])
        n = 1 << self.k
        self.advice, self.fixed, self.sigma = (self._columns(kind, n) for kind in range(3))
        p, cnt = C.POINTER(C.c_uint64)(), C.c_size_t()
        _check(_L().h2v_layout_instance(self._h, C.byref(p), C.byref(cnt)))
        self.instances = [np.ctypeslib.as_array(p, shape=(cnt.value, 4)).copy() if cnt.value else np.zeros((0, 4), dtype=np.uint64)]
        nb = C.c_size_t()
        _check(_L().h2v_layout_break_points(self._h, None, 0, C.byref(nb)))
        bp = np.zeros(max(1, nb.value), dtype=np.uint32)
        _check(_L().h2v_layout_break_points(self._h, _ptr(bp), bp.size, C.byref(nb)))
        self.break_points = [int(x) for x in bp[:nb.value]]
        G, Lc, NF = self.num_advice, self.num_lookup_advice, self.num_fixed
        A = G + Lc
        sel0 = 1 + NF
        self.cs = dict(
            k=self.k, degree=4, blinding_factors=self.BLINDING_FACTORS, n_advice=A, n_fixed=1 + NF + G, n_instance=1,
            gates=[(c, sel0 + c) for c in range(G)], lookups=[(G + l, 0) for l in range(Lc)],
            permutation=[(1, 1 + f) for f in range(NF)] + [(0, c) for c in range(A)] + [(2, 0)],
            advice_queries=[q for c in range(G) for q in ((c, 0), (c, 1), (c, 2), (c, 3))] + [(G + l, 0) for l in range(Lc)],
            fixed_queries=[(1 + f, 0) for f in range(NF)] + [(sel0 + c, 0) for c in range(G)] + [(0, 0)],
            instance_queries=[(0, 0)])

    def _columns(self, kind, n):
        pp, cnt = _u64pp(), C.c_size_t()
        _check(_L().h2v_layout_columns(self._h, kind, C.byref(pp), C.byref(cnt)))
        return [np.ctypeslib.as_array(pp[i], shape=(n, 4)) for i in range(cnt.value)]

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.advice = self.fixed = self.sigma = []
            _L().h2v_layout_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class WitnessProgram:
    """A recorded circuit compiled for replay on the GPU (h2v_witness_program_new): `generate(inputs_list)` gives, for
    each list of inputs (the values the recording passed to `assign_witnesses`, in that order, Montgomery limbs), the
    advice columns and instances `RangeCircuit(builder, k, minimum_rows)` would give for a builder run on those inputs.
    The recording's fixed and sigma columns serve them all.  The builder may be closed afterwards."""

    INFO = ("inputs", "cells", "computed_cells", "levels", "advice_columns", "instances", "k", "bytes_per_witness")

    def __init__(self, builder, k, minimum_rows=9):
        self._h = C.c_void_p()
        _check(_L().h2v_witness_program_new(builder._h, k, minimum_rows, C.byref(self._h)))
        out = np.zeros(8, dtype=np.uint64)
        _check(_L().h2v_witness_program_info(self._h, _ptr(out)))
        self.info = {name: int(v) for name, v in zip(self.INFO, out)}
        self.n_inputs, self.k = self.info["inputs"], self.info["k"]

    def inputs(self):
        """the recording's own inputs, (n_inputs, 4) Montgomery limbs"""
        out = np.zeros((self.n_inputs, 4), dtype=np.uint64)
        _check(_L().h2v_witness_program_inputs(self._h, _ptr(out)))
        return out

    def rule_counts(self):
        """computed cells per rule kind (zk_builder.hpp's RuleKind order)"""
        n = C.c_size_t()
        _check(_L().h2v_witness_program_rule_counts(self._h, None, 0, C.byref(n)))
        out = np.zeros(n.value, dtype=np.uint64)
        _check(_L().h2v_witness_program_rule_counts(self._h, _ptr(out), n.value, C.byref(n)))
        return [int(x) for x in out]

    def pack_inputs(self, inputs_list, who):
        """inputs_list as one (B, n_inputs, 4) array; errors start with `who`"""
        inp = np.zeros((len(inputs_list), self.n_inputs, 4), dtype=np.uint64)
        for w, x in enumerate(inputs_list):
            x = np.asarray(x, dtype=np.uint64).reshape(-1, 4)
            if x.shape[0] != self.n_inputs:
                raise ValueError(f"{who}: witness {w}: {x.shape[0]} inputs, the program has {self.n_inputs}")
            inp[w] = x
        return inp

    def generate(self, inputs_list):
        """-> [(advice, instances)] per witness, shaped like `RangeCircuit.advice` / `.instances`"""
        B = len(inputs_list)
        inp = self.pack_inputs(inputs_list, "witness_generate")
        n, A, I = 1 << self.k, self.info["advice_columns"], self.info["instances"]
        adv = np.zeros((B, A, n, 4), dtype=np.uint64)
        inst = np.zeros((B, I, 4), dtype=np.uint64)
        _check(_L().h2v_witness_generate(self._h, B, self.n_inputs, _ptr(inp), _ptr(adv), _ptr(inst)))
        return [([adv[w, c] for c in range(A)], [inst[w]]) for w in range(B)]

    @staticmethod
    def last_ms():
        """(upload, evaluation + gather, download) of the last generate, ms"""
        ms = (C.c_double * 3)()
        _check(_L().h2v_witness_last_ms(ms))
        return tuple(ms)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _L().h2v_witness_program_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------- the example circuits
def distance_functions(ctx, inp, make_public, fp=None):
    """/root/reference/examples/distances.rs:24-63"""
    a_in, b_in = inp["a"], inp["b"]
    if len(a_in) != len(b_in):
        raise ValueError("assertion failed: input.a.len() == input.b.len()")
    fp = fp or FixedPointChip.default(ctx.builder)
    dist = DistanceChip.default(fp)
    a = ctx.assign_witnesses(fp.quantize_vector(a_in))
    b = ctx.assign_witnesses(fp.quantize_vector(b_in))
    out = {}
    for name in ("euclidean", "manhattan", "cosine", "hamming"):
        d = getattr(dist, name + "_distance")(ctx, a, b)
        out[name] = fp.dequantization(d.value())
        make_public.append(d)
    return out


def exhaustive_merkle(ctx, inp, make_public, r_f=8, r_p=57, distance=DISTANCE_COSINE, fp=None):
    """/root/reference/examples/query.rs:32-73"""
    query_in, database_in = inp["query"], inp["database"]
    if any(len(v) != len(query_in) for v in database_in):
        raise ValueError("assertion failed: database vectors and query differ in length")
    fp = fp or FixedPointChip.default(ctx.builder)
    vdb = VectorDBChip.default(fp)
    poseidon = PoseidonChip(ctx, r_f, r_p)
    query = ctx.assign_witnesses(fp.quantize_vector(query_in))
    database = [ctx.assign_witnesses(fp.quantize_vector(v)) for v in database_in]
    _, result = vdb.nearest_vector(ctx, query, database, distance)
    make_public.extend(result)
    root = vdb.merkle_commitment(ctx, poseidon, database)
    make_public.append(root)
    return dict(result=fp.dequantize_vector(result), root=root.value())


def kmeans(ctx, inp, make_public, K=4, I=10, distance=DISTANCE_COSINE, fp=None):
    """/root/reference/examples/kmeans.rs:25-60"""
    vectors_in = inp["vectors"]
    if any(len(v) != len(vectors_in[0]) for v in vectors_in):
        raise ValueError("assertion failed: vectors differ in length")
    fp = fp or FixedPointChip.default(ctx.builder)
    vdb = VectorDBChip.default(fp)
    vectors = [ctx.assign_witnesses(fp.quantize_vector(v)) for v in vectors_in]
    centroids, indicators = vdb.kmeans(ctx, vectors, distance, K, I)
    for c in centroids:
        make_public.extend(c)
    return dict(centroids=[fp.dequantize_vector(c) for c in centroids], indicators=[fp.dequantize_vector(i) for i in indicators])


EXAMPLES = dict(distances=distance_functions, query=exhaustive_merkle, kmeans=kmeans)


def create_circuit(f, inp, k, lookup_bits, minimum_rows=9, record=False, **kw):
    """the scaffold's `create_circuit` (mod.rs:347-402): run the circuit function on `builder.main(0)`, expose the public
    values, lay the trace out.  Returns (RangeCircuit, whatever f returned); the circuit's `.builder` is a recording
    builder when record=True."""
    if not lookup_bits < k:
        raise ValueError("LOOKUP_BITS needs to be less than DEGREE")      # mod.rs:367
    builder = GateThreadBuilder(lookup_bits, record=record)
    public = []
    out = f(builder.main(0), inp, public, **kw)
    builder.make_public(public)
    return RangeCircuit(builder, k, minimum_rows), out


_PATTERN = [[1.123, 0.456, 0.789], [1.111, 0.111, 0.111], [0.111, 0.444, 1.777], [8.89, 4.456, 2.234]]


def example_input(name):
    """the inputs of the reference's examples (the values of /root/reference/data/{distances,query,kmeans}.in: two
    3-vectors; a query and the four-vector pattern repeated five times)"""
    if name == "distances":
        return dict(a=[0.123, 0.456, 1.789], b=[1.123, 0.456, 0.789])
    if name == "query":
        return dict(query=[0.123, 0.456, 1.789], database=[list(v) for _ in range(5) for v in _PATTERN])
    if name == "kmeans":
        return dict(vectors=[list(v) for _ in range(5) for v in _PATTERN])
    raise ValueError(name)


# BASELINE.json configs[0..2]: (k, LOOKUP_BITS) of the README's commands
EXAMPLE_PARAMS = dict(distances=(13, 12), query=(13, 12), kmeans=(16, 15))


def example_witness_inputs(name, inp, precision_bits=48):
    """the inputs the example circuit `name` assigns for `inp`, in assignment order: the `WitnessProgram` inputs of a
    recording of that example -> (n, 4) Montgomery limbs"""
    if name == "distances":
        leaves = list(inp["a"]) + list(inp["b"])
    elif name == "query":
        leaves = list(inp["query"]) + [x for v in inp["database"] for x in v]
    elif name == "kmeans":
        leaves = [x for v in inp["vectors"] for x in v]
    else:
        raise ValueError(name)
    b = GateThreadBuilder(EXAMPLE_PARAMS[name][1], precision_bits)
    try:
        return FixedPointChip.default(b).quantize_vector(leaves)
    finally:
        b.close()
