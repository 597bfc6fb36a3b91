"""GPU parity at the proof sizes (k = 17 to 20, extended columns up to 2^22 points) and the NTT sizes above them.

Every output of the kernels below is compared in full with the CPU oracle (or, for the host helpers, with Python big
integers), on seeded inputs from `O.fr_fill` in both of its modes (uniform; witness-like: zeros, ones, small values).
The sizes are the ones the small-size tests of test_gpu_parity.py / test_quotient.py cannot reach: the Montgomery NTT
kernel (L > 18) with several columns per launch, running products and kate division with more than 256 tiles per
scan, the quotient kernels with rotations that wrap a 2^22-point column, and the streamed permutation entry point."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from common import fr_arr, mem_available
from oracle import oracle as O
from oracle import pyref as P

pytestmark = pytest.mark.gpu

R = P.R
GIB = 1 << 30


def fe(x):
    return fr_arr([x])[0]


# ----------------------------------------------------------------------------- 1. best_fft at every large pass shape
@pytest.mark.parametrize("log_n", [20, 21, 22, 23, 24, 25])
def test_best_fft_large_vs_oracle(h2v, log_n):
    """best_fft at 2^20..2^25 in full: the Montgomery pass kernel (ntt_pass_kernel<false>) with the pass / tile shapes
    (7,7,6), (7,7,7), (8,7,7), (8,8,7), (8,8,8), (9,8,8); log_n = 21 also with another primitive root (omega^5)."""
    n = 1 << log_n
    a = O.fr_fill(n, 5000 + log_n, mode=log_n % 2)
    w = fe(P.omega_for(log_n))
    assert np.array_equal(h2v.best_fft(a, w, log_n), O.best_fft(a, w, log_n))
    if log_n == 21:
        w5 = fe(pow(P.omega_for(log_n), 5, R))
        assert np.array_equal(h2v.best_fft(a, w5, log_n), O.best_fft(a, w5, log_n))


@pytest.mark.parametrize("log_n", [26, 27])
def test_best_fft_largest_roundtrip(h2v, log_n):
    """best_fft at 2^26 and 2^27 (the largest sizes best_fft accepts): the forward transform with omega, then the
    inverse (the omega^-1 twiddle table and the 1/n post-scale of lagrange_to_coeff) gives back the whole input, and
    sampled outputs equal the polynomial evaluated at omega^j."""
    n = 1 << log_n
    if mem_available() < 5 * n * 32:
        pytest.skip(f"needs about {5 * n * 32 / GIB:.0f} GiB of free host memory")
    a = O.fr_fill(n, 6000 + log_n, mode=log_n % 2)
    wi = P.omega_for(log_n)
    out = h2v.best_fft(a, fe(wi), log_n)
    for j in (n - 1, random.Random(log_n).randrange(1, n - 1)):
        assert np.array_equal(out[j], O.fr_eval_poly(a, fe(pow(wi, j, R)))), j
    d = h2v.EvaluationDomain(2, log_n)           # k = extended_k = log_n: lagrange_to_coeff is the inverse best_fft
    assert np.array_equal(d.omega, fe(wi))
    back = d.lagrange_to_coeff(out)
    del out
    assert np.array_equal(back, a)
    d.close()


# ----------------------------------------------------------------------------- 2. EvaluationDomain at proof sizes
def _domain_ops_vs_oracle(h2v, j, k, seed):
    """all five ops and the fused divide-by-vanishing batch of EvaluationDomain(j, k), one column each"""
    d, od = h2v.EvaluationDomain(j, k), O.EvaluationDomain(j, k)
    assert d.extended_k == od.extended_k
    a = O.fr_fill(d.n, seed, mode=1)
    b = O.fr_fill(d.n, seed + 1, mode=0)
    e = O.fr_fill(d.extended_n, seed + 2, mode=seed % 2)
    assert np.array_equal(d.lagrange_to_coeff(a), od.lagrange_to_coeff(a))
    assert np.array_equal(d.coeff_to_lagrange(b), od.coeff_to_lagrange(b))
    assert np.array_equal(d.coeff_to_extended(a), od.coeff_to_extended(a))
    assert np.array_equal(d.extended_to_coeff(e), od.extended_to_coeff(e))
    dv = od.divide_by_vanishing_poly(e)
    assert np.array_equal(d.divide_by_vanishing_poly(e), dv)
    fused = d.transform_batch(h2v.OP_DIVIDE_BY_VANISHING, [e])[0]
    assert np.array_equal(fused, od.extended_to_coeff(dv))
    d.close()


@pytest.mark.parametrize("j,k", [(4, 17), (4, 18), (4, 19), (3, 18), (6, 18)])
def test_domain_ops_proof_sizes(h2v, j, k):
    """EvaluationDomain(j, k) ops in full at k = 17..19 (j = 4: extended 2^19..2^21, Montgomery kernel for every coset
    transform); j = 3 at k = 18 (extended_k = k + 1: no zero-padding shortcut); j = 6 at k = 18 (extended_k = k + 3,
    extended_to_coeff keeps 5n points, not a power of two).  k = 20 is in test_domain_ops_k20."""
    _domain_ops_vs_oracle(h2v, j, k, 100 * j + k)


K20_COLS = 4


@pytest.fixture(scope="module")
def k20():
    """EvaluationDomain(4, 20) inputs (4 columns of 2^20 and 4 of 2^22 points, both fill modes) and the oracle's outputs"""
    od = O.EvaluationDomain(4, 20)
    lag = [O.fr_fill(od.n, 2000 + i, mode=(i + 1) % 2) for i in range(K20_COLS)]
    ext = [O.fr_fill(1 << od.extended_k, 2100 + i, mode=i % 2) for i in range(K20_COLS)]
    want = {
        "l2c": [od.lagrange_to_coeff(c) for c in lag],
        "c2l": [od.coeff_to_lagrange(c) for c in lag],
        "c2e": [od.coeff_to_extended(c) for c in lag],
        "e2c": [od.extended_to_coeff(c) for c in ext],
        "fused": [od.extended_to_coeff(od.divide_by_vanishing_poly(c)) for c in ext],
    }
    return lag, ext, want


def test_domain_ops_k20(h2v, k20):
    """EvaluationDomain(4, 20) single-column ops in full: L = 20 (passes 7,7,6) for lagrange_to_coeff / coeff_to_lagrange,
    L = 22 (8,7,7) with the coset pre-scale, zero padding (pad4) and post-scales for the extended ops."""
    lag, ext, want = k20
    d, od = h2v.EvaluationDomain(4, 20), O.EvaluationDomain(4, 20)
    assert np.array_equal(d.lagrange_to_coeff(lag[0]), want["l2c"][0])
    assert np.array_equal(d.coeff_to_lagrange(lag[0]), want["c2l"][0])
    assert np.array_equal(d.coeff_to_extended(lag[0]), want["c2e"][0])
    assert np.array_equal(d.extended_to_coeff(ext[0]), want["e2c"][0])
    assert np.array_equal(d.divide_by_vanishing_poly(ext[1]), od.divide_by_vanishing_poly(ext[1]))
    assert np.array_equal(d.transform_batch(h2v.OP_DIVIDE_BY_VANISHING, [ext[0]])[0], want["fused"][0])
    d.close()


SENTINEL = np.uint64(0xA5A5A5A5A5A5A5A5)


def test_domain_transform_dev_k20_three_columns(h2v, k20):
    """transform_dev on 3 device-resident columns at k = 20 with a padded stride (2^22 + 8): the Montgomery kernel with
    blockIdx.y = 0, 1, 2 in every pass of every op.  The padding behind each output column is never written."""
    lag, ext, want = k20
    d = h2v.EvaluationDomain(4, 20)
    n, ne, cols = d.n, d.extended_n, 3
    stride = ne + 8
    d_in, d_out = h2v.DeviceBuffer(cols * stride * 32), h2v.DeviceBuffer(cols * stride * 32)
    fill = np.full((cols, stride, 4), SENTINEL, dtype=np.uint64)
    for op, inputs, key, nin, nout, work in ((h2v.OP_LAGRANGE_TO_COEFF, lag, "l2c", n, n, n),
                                             (h2v.OP_COEFF_TO_LAGRANGE, lag, "c2l", n, n, n),
                                             (h2v.OP_COEFF_TO_EXTENDED, lag, "c2e", n, ne, ne),
                                             (h2v.OP_EXTENDED_TO_COEFF, ext, "e2c", ne, 3 * n, ne),
                                             (h2v.OP_DIVIDE_BY_VANISHING, ext, "fused", ne, 3 * n, ne)):
        d_out.upload(fill)
        d_in.upload(fill)
        for c in range(cols):
            d_in.upload(inputs[c], offset=c * stride * 32)
        d.transform_dev(op, d_in.ptr, stride, d_out.ptr, stride, cols)
        got = d_out.download((cols, stride, 4))
        for c in range(cols):
            assert np.array_equal(got[c, :nout], want[key][c]), (key, c)
            assert (got[c, work:] == SENTINEL).all(), (key, c)
    d_in.free()
    d_out.free()
    d.close()


def test_domain_transform_batch_k20_pipelined(h2v, k20):
    """Host-facing transform_batch at k = 20 with 4 columns: every op runs as sub-batches of one column (32 to 128 MiB)
    rotating over the three upload / compute / download pipelines, the fourth column back on the first."""
    lag, ext, want = k20
    d = h2v.EvaluationDomain(4, 20)
    for op, inputs, key in ((h2v.OP_LAGRANGE_TO_COEFF, lag, "l2c"), (h2v.OP_COEFF_TO_LAGRANGE, lag, "c2l"),
                            (h2v.OP_COEFF_TO_EXTENDED, lag, "c2e"), (h2v.OP_EXTENDED_TO_COEFF, ext, "e2c"),
                            (h2v.OP_DIVIDE_BY_VANISHING, ext, "fused")):
        outs = d.transform_batch(op, inputs)
        for c in range(K20_COLS):
            assert np.array_equal(outs[c], want[key][c]), (key, c)
    d.close()


@pytest.mark.parametrize("j,k", [(4, 4), (2, 1)])
def test_domain_transform_dev_more_than_32768_columns(h2v, j, k):
    """40 000 columns in one transform_dev call: run_ntt launches them as 32 768 + 7 232, so the second chunk's
    column offsets are used (k = 4: one pass kernel; k = 1: the tiny kernel).  97 distinct columns repeat, and 97 does
    not divide 32 768, so a chunk that read or wrote the wrong columns would not match."""
    d, od = h2v.EvaluationDomain(j, k), O.EvaluationDomain(j, k)
    n, ne, cols, distinct = d.n, d.extended_n, 40000, 97
    base = np.stack([O.fr_fill(n, 7000 + i, mode=i % 2) for i in range(distinct)])
    idx = np.arange(cols) % distinct
    d_in, d_out = h2v.DeviceBuffer(cols * n * 32), h2v.DeviceBuffer(cols * ne * 32)
    d_in.upload(base[idx])
    for op, f, stride in ((h2v.OP_LAGRANGE_TO_COEFF, od.lagrange_to_coeff, n), (h2v.OP_COEFF_TO_EXTENDED, od.coeff_to_extended, ne)):
        d.transform_dev(op, d_in.ptr, n, d_out.ptr, stride, cols)
        got = d_out.download((cols, stride, 4))
        want = np.stack([f(c) for c in base])
        assert np.array_equal(got, want[idx]), op
    d_in.free()
    d_out.free()
    d.close()


@pytest.mark.parametrize("k", [0, 1, 2])
@pytest.mark.parametrize("j", [2, 3, 4, 9])
def test_domain_ops_small_domains(h2v, j, k):
    """Degenerate domains: k = 0..2 with j in {2, 3, 4, 9} gives transforms of 1 to 32 points -- the tiny kernel
    (L <= 2) with its table post-scale, and the single pass of L = 3..5 with zero padding."""
    _domain_ops_vs_oracle(h2v, j, k, 300 + 10 * j + k)


# ----------------------------------------------------------------------------- 3. running products, inversion, kate division
@pytest.mark.parametrize("n", [(1 << 19) + 1, 1 << 20, (1 << 21) + 3])
def test_grand_product_many_tiles(h2v, n):
    """grand_product with 257, 512 and 1025 tiles of 2048: fr_scan_top_kernel gives each thread 2 or 5 tiles (the last
    thread fewer); uniform numerators and denominators, and witness-like numerators."""
    num, den = O.fr_fill(n, 900 + n, mode=0), O.fr_fill(n, 901 + n, mode=0)
    assert np.array_equal(h2v.grand_product(num, den), O.fr_grand_product(num, den))
    num1 = O.fr_fill(n, 902 + n, mode=1)
    assert np.array_equal(h2v.grand_product(num1, den), O.fr_grand_product(num1, den))


def test_grand_product_dev_four_columns_k20(h2v):
    """grand_product_dev on 4 columns of 2^20 (one batch inversion for all, 512 tiles per column scan), with zero
    denominators in column 2 only: one early and two around the first tile boundary (2047, 2048)."""
    n, cols = 1 << 20, 4
    num = np.stack([O.fr_fill(n, 1100 + c, mode=c % 2) for c in range(cols)])
    den = np.stack([O.fr_fill(n, 1200 + c, mode=0) for c in range(cols)])
    den[2, [3, 2047, 2048]] = 0
    d_num, d_den, d_out = (h2v.DeviceBuffer(cols * n * 32) for _ in range(3))
    d_num.upload(num)
    d_den.upload(den)
    h2v.grand_product_dev(d_num.ptr, d_den.ptr, n, cols, d_out.ptr)
    got = d_out.download((cols, n, 4))
    for c in range(cols):
        assert np.array_equal(got[c], O.fr_grand_product(num[c], den[c])), c
    assert not got[2, 4:].any() and got[2, 3].any()
    for b in (d_num, d_den, d_out):
        b.free()


def test_batch_invert_2p20_with_zeros(h2v):
    """batch_invert at 2^20: a witness-like column (about 30 % zeros, ones, small values) and a uniform one with zeros
    at both ends and around a 2048 boundary; zeros stay zero."""
    n = 1 << 20
    a = O.fr_fill(n, 1300, mode=1)
    assert np.array_equal(h2v.batch_invert(a), O.fr_batch_invert(a))
    b = O.fr_fill(n, 1301, mode=0)
    b[[0, 2047, 2048, n - 1]] = 0
    assert np.array_equal(h2v.batch_invert(b), O.fr_batch_invert(b))


@pytest.mark.parametrize("n", [1 << 20, (1 << 21) + 5])
def test_kate_division_large(h2v, n):
    """kate_division and kate_division_dev at 2^20 and 2^21 + 5 coefficients (512 and 1025 tiles: the OpAdd scan with
    2 and 5 tiles per thread), for b != 0 and for b = 0 (the shift kernel)."""
    a = O.fr_fill(n, 1400 + n, mode=n % 2)
    d_a, d_q = h2v.DeviceBuffer(n * 32), h2v.DeviceBuffer((n - 1) * 32)
    d_a.upload(a)
    for b in (O.fr_fill(1, 1500 + n)[0], np.zeros(4, dtype=np.uint64)):
        want = O.fr_kate_division(a, b)
        assert np.array_equal(h2v.kate_division(a, b), want)
        h2v.kate_division_dev(d_a.ptr, n, b, d_q.ptr)
        assert np.array_equal(d_q.download((n - 1, 4)), want)
    d_a.free()
    d_q.free()


def test_eval_polynomial_quotient_piece_length(h2v):
    """eval_polynomial on 3 * 2^20 coefficients (the length of the quotient's pieces at k = 20, j = 4): 12 288
    coefficients per thread slice, at x = 0, 1, a root of unity and random points."""
    n = 3 << 20
    poly = O.fr_fill(n, 1600, mode=0)
    pts = np.concatenate([fr_arr([0, 1, P.omega_for(22)]), O.fr_fill(2, 1601)])
    got = h2v.eval_polynomial_batch([poly], pts)
    for i in range(len(pts)):
        assert np.array_equal(got[0, i], O.fr_eval_poly(poly, pts[i])), i


# ----------------------------------------------------------------------------- 4. quotient kernels at k = 18 and 20
class _Cols:
    """columns in one device allocation, `stride` elements apart, stored in `order` (slot of column c = order[c])"""

    def __init__(self, h2v, arrs, stride, order=None):
        self.stride = stride
        self.order = list(range(len(arrs))) if order is None else order
        self.buf = h2v.DeviceBuffer(max(1, len(arrs)) * stride * 32)
        for c, a in enumerate(arrs):
            self.buf.upload(a, offset=self.order[c] * stride * 32)

    def ptr(self, c=0):
        return self.buf.ptr + self.order[c] * self.stride * 32


def _ext_cols(ne, count, seed):
    return [O.fr_fill(ne, seed + i, mode=i % 2) for i in range(count)]


@pytest.mark.parametrize("k", [18, 20])
def test_quotient_gates_proof_sizes(h2v, k):
    """quotient_gates at k = 18 and 20 (2^20 / 2^22 rows, rotations 1..3 wrap the column end), 3 gates, padded strides."""
    gd, od = h2v.EvaluationDomain(4, k), O.EvaluationDomain(4, k)
    ne, gates = gd.extended_n, 3
    q, a = _ext_cols(ne, gates, 2200), _ext_cols(ne, gates, 2300)
    h0 = O.fr_fill(ne, 2400)
    y = O.fr_fill(1, 2401)[0]
    dq, da, dh = _Cols(h2v, q, ne + 8), _Cols(h2v, a, ne + 4), _Cols(h2v, [h0], ne)
    gd.quotient_gates(dh.ptr(), y, gates, dq.ptr(), ne + 8, da.ptr(), ne + 4)
    assert np.array_equal(dh.buf.download((ne, 4)), od.quotient_gates(h0, y, np.stack(q), np.stack(a)))
    gd.close()


@pytest.mark.parametrize("k", [18, 20])
def test_quotient_lookup_proof_sizes(h2v, k):
    """quotient_lookup at k = 18 and 20: the rotations +1 and -1 wrap a 2^20 / 2^22-row column."""
    gd, od = h2v.EvaluationDomain(4, k), O.EvaluationDomain(4, k)
    ne = gd.extended_n
    arrs = _ext_cols(ne, 8, 2500)        # input, table, A', S', z, l0, l_last, l_active
    h0 = O.fr_fill(ne, 2600)
    y, beta, gamma = O.fr_fill(3, 2601)
    d, dh = _Cols(h2v, arrs, ne), _Cols(h2v, [h0], ne)
    gd.quotient_lookup(dh.ptr(), y, beta, gamma, *[d.ptr(i) for i in range(8)])
    assert np.array_equal(dh.buf.download((ne, 4)), od.quotient_lookup(h0, y, beta, gamma, *arrs))
    gd.close()


PERM_COLS, PERM_CHUNK, PERM_BF = 5, 2, 5          # 3 sets, the last one of a single column


@pytest.fixture(scope="module", params=[18, 20])
def perm_case(request):
    """random extended columns of a 5-column permutation argument (degree 4: chunk 2, 3 sets) and the oracle's h"""
    k = request.param
    od = O.EvaluationDomain(4, k)
    ne = 1 << od.extended_k
    n_sets = (PERM_COLS + PERM_CHUNK - 1) // PERM_CHUNK
    cols, sigma, z = _ext_cols(ne, PERM_COLS, 2700), _ext_cols(ne, PERM_COLS, 2800), _ext_cols(ne, n_sets, 2900)
    l0, ll, la, h0 = _ext_cols(ne, 4, 3000)
    y, beta, gamma = O.fr_fill(3, 3100 + k)
    want = od.quotient_permutation(h0, y, beta, gamma, PERM_CHUNK, np.stack(cols), np.stack(sigma), np.stack(z), l0, ll, la, PERM_BF)
    return dict(k=k, ne=ne, n_sets=n_sets, cols=cols, sigma=sigma, z=z, l=[l0, ll, la], h0=h0, y=y, beta=beta, gamma=gamma,
                want=want)


def test_quotient_permutation_proof_sizes(h2v, perm_case):
    """quotient_permutation (strided columns) at k = 18 and 20: 5 columns in 3 sets, the last rotation
    -(blinding_factors + 1) wraps the column start."""
    pc = perm_case
    gd, ne = h2v.EvaluationDomain(4, pc["k"]), pc["ne"]
    dc, ds, dz = _Cols(h2v, pc["cols"], ne), _Cols(h2v, pc["sigma"], ne + 4), _Cols(h2v, pc["z"], ne + 8)
    dl, dh = _Cols(h2v, pc["l"], ne), _Cols(h2v, [pc["h0"]], ne)
    gd.quotient_permutation(dh.ptr(), pc["y"], pc["beta"], pc["gamma"], PERM_COLS, PERM_CHUNK, dc.ptr(), ne, ds.ptr(), ne + 4,
                            dz.ptr(), ne + 8, dl.ptr(0), dl.ptr(1), dl.ptr(2), PERM_BF)
    assert np.array_equal(dh.buf.download((ne, 4)), pc["want"])
    gd.close()


@pytest.mark.parametrize("ranges", [
    [(0, 3)],                       # all sets at once
    [(0, 1), (1, 2), (2, 3)],       # one set per call
    [(0, 0), (0, 1), (1, 3)],       # the head alone first, then uneven ranges
    [(0, 2), (2, 2), (2, 3)],       # an empty range in the middle
], ids=["all", "one-per-call", "head-alone", "empty-middle"])
def test_quotient_permutation_range_ptrs(h2v, perm_case, ranges):
    """h2v_quotient_permutation_range_ptrs_dev, the entry point of the streamed k = 20 prover, at k = 18 and 20: the sets
    split into consecutive ranges, columns through device pointer tables (stored in reverse order in HBM, so only the
    table says where a column is), with_head on the first call only.  The folded h equals the oracle's single call."""
    pc = perm_case
    gd, ne = h2v.EvaluationDomain(4, pc["k"]), pc["ne"]
    rev = list(range(PERM_COLS - 1, -1, -1))
    dc, ds = _Cols(h2v, pc["cols"], ne, rev), _Cols(h2v, pc["sigma"], ne, rev)
    dz, dl, dh = _Cols(h2v, pc["z"], ne + 8), _Cols(h2v, pc["l"], ne), _Cols(h2v, [pc["h0"]], ne)
    tables = []
    for t, (s0, s1) in enumerate(ranges):
        c0, c1 = min(PERM_COLS, s0 * PERM_CHUNK), min(PERM_COLS, s1 * PERM_CHUNK)
        tab = []
        for cols in (dc, ds):
            ptrs = np.array([cols.ptr(c) for c in range(c0, c1)] or [0], dtype=np.uint64)
            b = h2v.DeviceBuffer(ptrs.nbytes)
            b.upload(ptrs)
            tab.append(b)
        tables += tab
        gd.quotient_permutation_range(dh.ptr(), pc["y"], pc["beta"], pc["gamma"], PERM_COLS, PERM_CHUNK, s0, s1, t == 0,
                                      tab[0].ptr, tab[1].ptr, dz.ptr(), ne + 8, dl.ptr(0), dl.ptr(1), dl.ptr(2), PERM_BF)
    assert np.array_equal(dh.buf.download((ne, 4)), pc["want"])
    for b in tables:
        b.free()
    gd.close()


# ----------------------------------------------------------------------------- 5. NTT knobs
KNOB_FFT_LOG_NS = [3, 9, 10, 17, 18, 19, 22]
KNOB_DOMAIN_KS = [3, 10, 16, 20]


@pytest.fixture(scope="module")
def knob_oracle():
    inputs, want = {}, {}
    for log_n in KNOB_FFT_LOG_NS:
        a, w = O.fr_fill(1 << log_n, 3200 + log_n, mode=log_n % 2), fe(P.omega_for(log_n))
        inputs[f"fft_a_{log_n}"], inputs[f"fft_w_{log_n}"] = a, w
        want[f"fft_{log_n}"] = O.best_fft(a, w, log_n)
    for k in KNOB_DOMAIN_KS:
        od = O.EvaluationDomain(4, k)
        a, e = O.fr_fill(od.n, 3300 + k, mode=1), O.fr_fill(1 << od.extended_k, 3400 + k)
        inputs[f"dom_a_{k}"], inputs[f"dom_e_{k}"] = a, e
        want[f"l2c_{k}"], want[f"c2l_{k}"] = od.lagrange_to_coeff(a), od.coeff_to_lagrange(a)
        want[f"c2e_{k}"], want[f"e2c_{k}"] = od.coeff_to_extended(a), od.extended_to_coeff(e)
        want[f"dvp_{k}"] = od.divide_by_vanishing_poly(e)
        want[f"fused_{k}"] = od.extended_to_coeff(want[f"dvp_{k}"])
    return inputs, want


@pytest.mark.parametrize("knob,value", [("H2V_NTT_LOGE", "9"), ("H2V_NTT_LOGE", "10"), ("H2V_NTT_LOGE", "11"),
                                        ("H2V_NTT_SHOUP_MAX_L", "0"), ("H2V_NTT_SHOUP_MAX_L", "30")])
def test_ntt_knobs_change_the_schedule_not_the_result(knob_oracle, tmp_path, knob, value):
    """The NTT schedule knobs are read once per process, so a child process runs with each setting: H2V_NTT_LOGE = 9
    (tiles of T = 1 when a pass has S = 9 stages), 10, 11 (2048-element tiles); H2V_NTT_SHOUP_MAX_L = 0 (Montgomery
    kernel at every size) and 30 (Shoup kernel up to 2^22).  best_fft at 2^3..2^22 and the domain ops at k = 3, 10, 16,
    20 must equal the oracle.  Only the child's environment is set."""
    inputs, want = knob_oracle
    np.savez(tmp_path / "inputs.npz", **inputs)
    env = {kv: v for kv, v in os.environ.items() if kv not in ("H2V_NTT_LOGE", "H2V_NTT_SHOUP_MAX_L")}
    env[knob] = value
    child = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ntt_knob_child.py")
    res = subprocess.run([sys.executable, child, str(tmp_path)], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    with np.load(tmp_path / "outputs.npz") as got:
        assert sorted(got.files) == sorted(want)
        for key in want:
            assert np.array_equal(got[key], want[key]), key
    os.remove(tmp_path / "inputs.npz")
    os.remove(tmp_path / "outputs.npz")


# ----------------------------------------------------------------------------- 6. domain host helpers
@pytest.mark.parametrize("j,k", [(4, 5), (3, 7), (4, 20)])
def test_domain_host_helpers(h2v, j, k):
    """rotate_omega, rotate_extended, l_i_range and the empty / constant fills against Python big integers
    (oracle/pyref.py): positive and negative rotations, shifts that wrap past the column length, x on the domain."""
    d, pd = h2v.EvaluationDomain(j, k), P.Domain(j, k)
    n, ne = d.n, d.extended_n
    per = ne // n
    rnd = random.Random(1000 * j + k)
    w = pd.omega
    assert O.fr_to_ints(d.omega) == [w]
    # rotate_omega(value, rot) = value * omega^rot
    v = rnd.randrange(R)
    for rot in (0, 1, -1, 3, -5, n - 1, -(n + 7), 2 ** 31 - 1, -(2 ** 31)):
        assert O.fr_to_ints(d.rotate_omega(fe(v), rot)) == [v * pow(w, rot, R) % R], rot
    # rotate_extended(poly, rot)[i] = poly[(i + rot * 2^(extended_k - k)) mod 2^extended_k]
    poly = O.fr_fill(ne, 3500 + k)
    for rot in (0, 1, -1, -3, n // 2 + 1, n + 3, -(n + 5), 5 * n - 2, -(2 ** 31), 2 ** 31 - 1):
        idx = np.array([(i + rot * per) % ne for i in range(ne)]) if ne <= 1 << 12 else (np.arange(ne, dtype=np.int64) + rot * per) % ne
        assert np.array_equal(d.rotate_extended(poly, rot), poly[idx]), rot
    # l_i_range(x, xn, lo..hi)[t] = omega^i (xn - 1) / (n (x - omega^i)), i = lo + t; 0 where x = omega^i
    ninv = pow(n, -1, R)

    def l_i(x, xn, i):
        wi = pow(w, i, R)
        den = (x - wi) % R
        return wi * (xn - 1) * ninv * (pow(den, -1, R) if den else 0) % R

    x = rnd.randrange(R)
    for x_, xn in ((x, pow(x, n, R)), (x, rnd.randrange(R)), (pow(w, 2, R), 1), (pow(w, 2, R), rnd.randrange(R)),
                   (pow(w, -1, R), rnd.randrange(R))):
        for lo, hi in ((-3, 5), (0, 1), (-7, -2), (n - 2, n + 2)):
            got = d.l_i_range(fe(x_), fe(xn), range(lo, hi))
            assert O.fr_to_ints(got) == [l_i(x_, xn, i) for i in range(lo, hi)], (lo, hi)
    # fills
    s = fe(rnd.randrange(R))
    for arr, length in ((d.empty_coeff(), n), (d.empty_lagrange(), n), (d.empty_extended(), ne)):
        assert arr.shape == (length, 4) and not arr.any()
    for arr, length in ((d.constant_lagrange(s), n), (d.constant_extended(s), ne)):
        assert arr.shape == (length, 4) and (arr == s).all()
    d.close()
