"""The two batched device paths a proof spends its time in, bit for bit at the shapes of the kmeans (k = 16) and SIFT
(k = 20) proofs that bench.py times.

MSM commit batches (run_msm): 617 distinct columns at k = 16 (the kmeans proof's advice count) and 361 at k = 20 (one
more than the SIFT proof's commitments), so that the batch splits into several launches with a ragged last one; both
bases; column counts that move the bucket reduction's schedule; and, in a child process each, the scatter-slice, window
and chunk knobs.  Every commitment is compared with the oracle's closed form (sum_i s_i (a i + b)) G of the bases used.

Lookup batch (run_permute_batch): 72 lookups over one table at k = 16, 8 lookups over two tables at k = 20, a batch of
edge cases at u = 2^16 and 2^16 + 1, and batches with a value missing from the table.  Every lookup's A' and S' is
compared with the oracle's permute_expression_pair, one lookup at a time.

Smaller batches of the same entry points are in test_gpu_parity.py and test_lookup.py."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from common import fr_arr, mem_available
from halo2_vectordb_b200.circuit import RangeCircuit
from oracle import oracle as O
from oracle import pyref as P

pytestmark = pytest.mark.gpu

R = P.R
GIB = 1 << 30
SENTINEL = np.uint64(0xA5A5A5A5A5A5A5A5)
LAGRANGE, MONOMIAL = 1, 0                          # H2V_BASIS_LAGRANGE, H2V_BASIS_MONOMIAL
AB_LAGRANGE = (0x9E3779B97F4A7C15 >> 2, 0x632BE59BD9B4E019 >> 2)      # O.gen_bases' defaults
AB_MONOMIAL = (12345677, 987654321)
WORKERS = max(1, min(8, os.cpu_count() or 1))
TAIL = 8                                           # sentinel rows behind the last commitment


def _need_host(nbytes):
    if mem_available() < nbytes:
        pytest.skip(f"needs about {nbytes / GIB:.1f} GiB of free host memory")


# ----------------------------------------------------------------------------- 1. MSM commit batches
@pytest.fixture(scope="module")
def srs16(h2v):
    srs = h2v.ParamsKZG(16, None, O.gen_bases(1 << 16))
    srs.main_window = srs.info()                   # before any commit: (c, W) of the table the cost model picks
    yield srs
    srs.close()


@pytest.fixture(scope="module")
def srs20(h2v):
    n = 1 << 20
    srs = h2v.ParamsKZG(20, O.gen_bases(n, *AB_MONOMIAL), O.gen_bases(n, *AB_LAGRANGE))
    srs.main_window = srs.info()
    yield srs
    srs.close()


def _upload_columns(h2v, n, count, stride, make, bases=(AB_LAGRANGE,)):
    """Column i = make(i) of `count` columns is generated on the host (one per worker thread at a time), uploaded to one
    device buffer at element i * stride and dropped.  Returns the buffer and, for each (a, b) of `bases`, the (count, 8)
    closed forms of the columns."""
    buf = h2v.DeviceBuffer(count * stride * 32)
    want = np.zeros((len(bases), count, 8), dtype=np.uint64)

    def one(i):
        col = make(i)
        for j, (a, b) in enumerate(bases):
            want[j, i] = O.msm_closed_form(col, a=a, b=b)
        buf.upload(col, offset=i * stride * 32)

    with ThreadPoolExecutor(WORKERS) as ex:
        list(ex.map(one, range(count)))
    return buf, want


def _commit_checked(h2v, srs, d_cols, stride, count, n, want, basis=LAGRANGE):
    """commit_batch_dev of `count` columns into an output buffer filled with a sentinel: every commitment equals `want`,
    and the TAIL rows behind the last one are never written"""
    d_out = h2v.DeviceBuffer((count + TAIL) * 64)
    d_out.upload(np.full((count + TAIL, 8), SENTINEL, dtype=np.uint64))
    srs.commit_batch_dev(d_cols.ptr, stride, count, n, d_out.ptr, basis=basis)
    got = d_out.download((count + TAIL, 8))
    d_out.free()
    bad = [i for i in range(count) if not np.array_equal(got[i], want[i])]
    assert not bad, f"{len(bad)} of {count} commitments differ from the closed form: columns {bad[:64]} (last table {srs.info()})"
    assert (got[count:] == SENTINEL).all(), "commit_batch_dev wrote past its last commitment"


def _witness_or_uniform(n, seed, witness, lookup_bits):
    return O.fr_fill(n, seed, mode=1 if witness else 0, lookup_bits=lookup_bits)


def _k20_column(i, n):
    """column i of the 361-column batch: a special column every 17th slot (all zero, all one, all r - 1, non-zero on row
    n - 1 only), witness-like (lookup_bits = 19: giant buckets) every third, uniform otherwise"""
    if i % 17 == 0:
        kind = (i // 17) % 4
        if kind == 0:
            return np.zeros((n, 4), dtype=np.uint64)
        if kind in (1, 2):
            return np.tile(fr_arr([1 if kind == 1 else R - 1]), (n, 1))
        col = np.zeros((n, 4), dtype=np.uint64)
        col[n - 1] = O.fr_fill(1, 30000 + i)[0]
        return col
    return _witness_or_uniform(n, 20000 + i, i % 3 == 1, 19)


def test_commit_k20_sift_batch_splits_into_launches(h2v, srs20):
    """361 distinct device-resident columns of 2^20 at a padded stride (2^20 + 8) in one commit_batch_dev call.  No launch
    can hold them: W = ceil(255 / c) >= 11 windows for every window WindowDispatch instantiates (c <= 24), and 361 * 11
    * 2^20 entries exceed run_msm's 2^31 limit, so its launch split runs -- several launches, each writing its results at
    d_out_aff + c0, the last one ragged -- with distinct special columns (every 17th) on both sides of any boundary.
    test_large_batches_take_the_pipelined_paths splits 700 copies of ONE 2^16 column (stride 0), test_commit_k20_closed_form
    commits 2 columns of 2^20: neither can tell a launch that reads or writes another launch's columns."""
    n, count = 1 << 20, 361
    stride = n + 8
    assert all(count * ((255 + c - 1) // c) * n >= 1 << 31 for c in range(3, 25))
    _need_host(WORKERS * 4 * n * 32 + GIB // 2)
    d_cols, want = _upload_columns(h2v, n, count, stride, lambda i: _k20_column(i, n))
    try:
        _commit_checked(h2v, srs20, d_cols, stride, count, n, want[0])
    finally:
        d_cols.free()


def test_commit_k16_kmeans_batch_distinct_columns(h2v, srs16):
    """617 distinct columns of 2^16 (the kmeans proof's advice count, as in bench.py's kmeans-shaped proof), uniform and
    witness-like (lookup_bits = 15) alternating, in one commit_batch_dev call: one launch with n_inst = 617 reduction
    instances.
    test_large_batches_take_the_pipelined_paths commits 700 copies of one column, so a launch that mixed up columns or
    their results would still pass it."""
    n, count = 1 << 16, 617
    d_cols, want = _upload_columns(h2v, n, count, n, lambda i: _witness_or_uniform(n, 16000 + i, i % 2 == 1, 15))
    try:
        _commit_checked(h2v, srs16, d_cols, n, count, n, want[0])
    finally:
        d_cols.free()


def test_commit_k20_both_bases(h2v, srs20):
    """5 columns of 2^20 through both bases of one SRS handle built from two different base sets: the monomial basis's
    window tables (commit_batch_dev(..., basis=MONOMIAL)) against the closed form of (a_m i + b_m) G, the Lagrange basis's
    against the default (a, b).  test_commit_vs_closed_form checks the monomial basis with single columns up to 2^16 only."""
    n, count = 1 << 20, 5
    _need_host(WORKERS * 4 * n * 32 + GIB // 2)
    d_cols, want = _upload_columns(h2v, n, count, n, lambda i: _k20_column(i + 1, n), bases=(AB_LAGRANGE, AB_MONOMIAL))
    try:
        _commit_checked(h2v, srs20, d_cols, n, count, n, want[0], basis=LAGRANGE)
        _commit_checked(h2v, srs20, d_cols, n, count, n, want[1], basis=MONOMIAL)
    finally:
        d_cols.free()


@pytest.fixture(scope="module")
def k20_columns(h2v):
    """45 device-resident uniform columns of 2^20 and their closed forms"""
    n, count = 1 << 20, 45
    _need_host(WORKERS * 4 * n * 32 + GIB // 2)
    d_cols, want = _upload_columns(h2v, n, count, n, lambda i: O.fr_fill(n, 21000 + i))
    yield d_cols, want[0]
    d_cols.free()


@pytest.mark.parametrize("count", [1, 2, 3, 45])
def test_commit_k20_reduction_schedule(h2v, srs20, k20_columns, count):
    """The first 1, 2, 3 and 45 of 45 uniform columns of 2^20 in one launch: the bucket reduction runs n_inst = count
    instances (one group per column with the precomputed tables).  msm_srs weighs the reduction up for batches of fewer
    than 32 columns, so 1 to 3 columns take the small window (2^17 buckets): with n_inst * 128 below 148 * 256 partial
    sums the second serial level of msm_reduce_kernel shortens its segments to 8 (log_seg = 3) before msm_reduce_tree_kernel
    takes the last 512.  45 columns take the main window (2^19 buckets) and keep segments of 32 on both serial levels.
    test_commit_k20_closed_form runs 2 columns only, through the host-facing entry point."""
    d_cols, want = k20_columns
    n = 1 << 20
    _commit_checked(h2v, srs20, d_cols, n, count, n, want[:count])


KNOB_COLS = {16: 33, 20: 7}
KNOBS = ("H2V_SCATTER_SLICES", "H2V_RED_WEIGHT", "H2V_CHUNK")


@pytest.fixture(scope="module")
def knob_case(tmp_path_factory):
    """inputs.npz for msm_knob_child.py (33 columns of 2^16, 7 of 2^20, uniform and witness-like alternating) and the
    closed forms of the commitments the child writes"""
    _need_host(GIB)
    work = tmp_path_factory.mktemp("msm_knobs")
    inputs, want = {}, {}
    for k, count in KNOB_COLS.items():
        n = 1 << k
        cols = np.stack([_witness_or_uniform(n, 40000 + 100 * k + i, i % 2 == 1, k - 1) for i in range(count)])
        inputs[f"cols_{k}"] = cols
        want[f"commit_{k}"] = np.stack([O.msm_closed_form(c) for c in cols])
    want["commit_20_one"] = want["commit_20"][1:2]
    np.savez(work / "inputs.npz", **inputs)
    return work, want


@pytest.mark.parametrize("knob,value", [("H2V_SCATTER_SLICES", "2"), ("H2V_SCATTER_SLICES", "3"), ("H2V_SCATTER_SLICES", "7"),
                                        ("H2V_RED_WEIGHT", "0.5"), ("H2V_RED_WEIGHT", "50"),
                                        ("H2V_CHUNK", "12"), ("H2V_CHUNK", "64")])
def test_msm_knobs_change_the_schedule_not_the_result(srs16, srs20, knob_case, tmp_path, knob, value):
    """The MSM knobs are read once per process, so a child process (msm_knob_child.py) runs with each setting and commits
    33 columns of 2^16, 7 of 2^20 and 1 of 2^20 device-resident; every commitment must equal the closed form.

    H2V_SCATTER_SLICES = 2, 3, 7: run_msm's slice loop with an uneven `per` and a last slice clipped by min(sh.nb, ...),
    also on batches of several columns (by default only a single column of >= 1 GiB of entries is sliced, in 4:
    test_best_multiexp_sweep_sizes_closed_form at 2^24).  H2V_RED_WEIGHT = 0.5 and 50: choose_cfg picks a larger window
    (c = 17 at 2^16, 22 at 2^20) and a smaller one (13 at 2^16, 16 at 2^20) than by default, so other WindowDispatch<C>
    instantiations and their precomputed tables run at proof size; the child's main table must differ from this process's
    (a weight of 1 would keep c = 20 at 2^20).  The other knobs must leave the window alone.  H2V_CHUNK = 12 and 64: the
    accumulate chunk at both ends of pick_chunk's clamp (test_msm_tuning_invariance forces chunks at 2^11 only).
    Only the child's environment is set."""
    work, want = knob_case
    env = {kv: v for kv, v in os.environ.items() if kv not in KNOBS}
    env[knob] = value
    child = os.path.join(os.path.dirname(os.path.abspath(__file__)), "msm_knob_child.py")
    res = subprocess.run([sys.executable, child, str(work), str(tmp_path)], env=env, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout + res.stderr
    with np.load(tmp_path / "outputs.npz") as got:
        for key in want:
            bad = [i for i in range(len(want[key])) if not np.array_equal(got[key][i], want[key][i])]
            assert not bad, (key, bad)
        for k, srs in ((16, srs16), (20, srs20)):
            window = tuple(int(x) for x in got[f"window_{k}"])
            if knob == "H2V_RED_WEIGHT":
                assert window != srs.main_window, (k, window)
            else:
                assert window == srs.main_window, (k, window)


# ----------------------------------------------------------------------------- 2. lookup batch
def _mont(values):
    """small non-negative integers (u64) -> Montgomery Fr rows"""
    v = np.asarray(values, dtype=np.uint64)
    z = np.zeros_like(v)
    return O.to_mont(np.stack([v, z, z, z], axis=1))


def _range_table(bits, u):
    """halo2-base's range table: 0 .. 2^bits - 1, the remaining usable rows zero"""
    return _mont(np.concatenate([np.arange(1 << bits, dtype=np.uint64), np.zeros(u - (1 << bits), dtype=np.uint64)]))


class _Lookups:
    """A batch of lookups on the device: input l (Montgomery, `u` rows) is looked up in tables[which[l]].  The inputs sit in
    one buffer (every pointer distinct), each distinct table once (lookups of one table share its pointer, so it is sorted
    once).  The oracle's A', S' of every lookup are computed up front; the host inputs are not kept."""

    def __init__(self, h2v, inputs, tables, which, stride):
        self.h2v, self.which, self.stride = h2v, list(which), stride
        self.L, self.u = len(inputs), inputs[0].shape[0]
        u = self.u
        self.want = [O.permute_expression_pair(inputs[l], tables[w]) for l, w in enumerate(which)]
        self.d_in, self.d_tab = h2v.DeviceBuffer(self.L * u * 32), h2v.DeviceBuffer(len(tables) * u * 32)
        for l, v in enumerate(inputs):
            self.d_in.upload(v, offset=l * u * 32)
        for t, v in enumerate(tables):
            self.d_tab.upload(v, offset=t * u * 32)
        self.in_ptrs = [self.d_in.ptr + l * u * 32 for l in range(self.L)]
        self.tab_ptrs = [self.d_tab.ptr + w * u * 32 for w in which]
        self.d_a, self.d_s = h2v.DeviceBuffer(self.L * stride * 32), h2v.DeviceBuffer(self.L * stride * 32)

    def run(self, in_ptrs=None):
        """one permute_expression_pair_batch_dev call into outputs filled with the sentinel first"""
        fill = np.full((self.L * self.stride, 4), SENTINEL, dtype=np.uint64)
        self.d_a.upload(fill)
        self.d_s.upload(fill)
        del fill
        self.h2v.permute_expression_pair_batch_dev(in_ptrs or self.in_ptrs, self.tab_ptrs, self.u, self.d_a.ptr, self.stride,
                                                   self.d_s.ptr, self.stride)

    def check(self, what=""):
        """A' and S' of every lookup equal the oracle's; the padding rows u .. stride of each output are never written"""
        u, stride = self.u, self.stride
        for l in range(self.L):
            for name, buf, want in (("A'", self.d_a, self.want[l][0]), ("S'", self.d_s, self.want[l][1])):
                got = buf.download((stride, 4), offset=l * stride * 32)
                bad = np.flatnonzero((got[:u] != want).any(axis=1))
                assert bad.size == 0, f"{what} lookup {l} of {self.L} (table {self.which[l]}): {name} differs on {bad.size} rows, first {bad[:16]}"
                assert (got[u:] == SENTINEL).all(), f"{what} lookup {l}: {name} written past row u = {u}"

    def free(self):
        for b in (self.d_in, self.d_tab, self.d_a, self.d_s):
            b.free()


KMEANS_K, KMEANS_LOOKUPS, KMEANS_BITS = 16, 72, 15
SIFT_K, SIFT_LOOKUPS, SIFT_BITS = 20, 8, 19


def _usable_rows(k):
    """rows a lookup argument permutes: n minus the blinding rows and the last row (RangeCircuit's constraint system)"""
    return (1 << k) - (RangeCircuit.BLINDING_FACTORS + 1)


def _range_input(rng, bits, u, l):
    """range-check values of lookup l: uniform; mostly zero; small (few distinct values, long runs of repeats)"""
    kind = l % 3
    if kind == 0:
        return rng.integers(0, 1 << bits, u, dtype=np.uint64)
    if kind == 1:
        v = rng.integers(0, 1 << bits, u, dtype=np.uint64)
        v[rng.random(u) < 0.6] = 0
        return v
    return rng.integers(0, 1 << 8, u, dtype=np.uint64)


@pytest.fixture(scope="module")
def kmeans_lookups(h2v):
    """the kmeans proof's lookup batch: 72 lookups (about as many as the proof has) of 2^16 - 7 usable rows over one range
    table 0 .. 2^15 - 1"""
    u = _usable_rows(KMEANS_K)
    rng = np.random.default_rng(72)
    inputs = [_mont(_range_input(rng, KMEANS_BITS, u, l)) for l in range(KMEANS_LOOKUPS)]
    lk = _Lookups(h2v, inputs, [_range_table(KMEANS_BITS, u)], [0] * KMEANS_LOOKUPS, 1 << KMEANS_K)
    del inputs
    yield lk
    lk.free()


def test_lookup_batch_kmeans_shape(kmeans_lookups):
    """72 lookups x (2^16 - 7) rows over ONE table pointer (sorted once: 73 key slices), outputs at stride 2^16 as the
    prover lays them out: the flags of all lookups scanned as one array of 4.7 M entries (2304 scan tiles), and
    lookup_emit_table_batch_kernel's non-last lookups (leftover counts from rep_offs[row0 + u] - rep_offs[row0]) and last
    lookup (from totals).  test_gpu_permute_batch_matches_per_lookup_oracle runs 5 lookups of at most 5000 rows."""
    kmeans_lookups.run()
    kmeans_lookups.check("kmeans")


def test_lookup_batch_errors_leave_the_context_usable(kmeans_lookups):
    """A value outside the table (2^15, above its largest entry) in the FIRST lookup only, then a full-width value (r - 1)
    in the LAST lookup only, of the kmeans batch: each call raises ValueError, and after each the device's lookup context
    gives the right A', S' for the good batch again.  test_gpu_permute_batch_matches_per_lookup_oracle puts a bad value
    in a middle lookup and never calls again."""
    lk, h2v, u = kmeans_lookups, kmeans_lookups.h2v, kmeans_lookups.u
    for l, bad_value in ((0, fr_arr([1 << KMEANS_BITS])[0]), (lk.L - 1, fr_arr([R - 1])[0])):
        col = lk.d_in.download((u, 4), offset=l * u * 32)
        col[u // 2] = bad_value
        d_bad = h2v.DeviceBuffer(u * 32)
        d_bad.upload(col)
        ptrs = list(lk.in_ptrs)
        ptrs[l] = d_bad.ptr
        with pytest.raises(ValueError):
            lk.run(ptrs)
        d_bad.free()
        lk.run()
        lk.check(f"after a missing value in lookup {l}:")


def test_lookup_batch_sift_shape(h2v):
    """8 lookups x (2^20 - 7) rows over 2 distinct tables (LOOKUP_BITS = 19) interleaved as 1 0 0 1 0 1 1 0, so the
    lookups' table slices (tmap) are not monotone: table 0 is the range table, table 1 the values 3 i + 5 padded with 5
    and shuffled.  8.4 M flags in one scan, 10 key slices of 2^20 in every bitonic launch.  test_gpu_permute_k20_properties
    _and_dev_entry permutes one lookup of this size."""
    u = _usable_rows(SIFT_K)
    _need_host(2 * GIB)
    rng = np.random.default_rng(20)
    t1 = np.concatenate([3 * np.arange(1 << SIFT_BITS, dtype=np.uint64) + 5, np.full(u - (1 << SIFT_BITS), 5, dtype=np.uint64)])
    tables = [_range_table(SIFT_BITS, u), _mont(rng.permutation(t1))]
    which = [1, 0, 0, 1, 0, 1, 1, 0]
    inputs = []
    for l, w in enumerate(which):
        v = _range_input(rng, SIFT_BITS, u, l)
        inputs.append(_mont(3 * v + 5 if w else v))
    lk = _Lookups(h2v, inputs, tables, which, (1 << SIFT_K) + 4)
    del inputs, tables
    try:
        lk.run()
        lk.check("sift")
    finally:
        lk.free()


def _wide_families(rng, count):
    """2 * count canonical full-width values: `count` that differ only in bits 224..255 (the 32-bit limb key_less compares
    first) and `count` that differ only in bits 0..31 (the limb it compares last); all below r"""
    base = rng.integers(0, 1 << 63, 3, dtype=np.uint64)
    top = np.tile(np.append(base, np.uint64(0x12345678)), (count, 1))
    top[:, 3] += np.arange(1, count + 1, dtype=np.uint64) << np.uint64(32)
    low = np.tile(np.append(base, np.uint64(0x30644E70 << 32)), (count, 1))
    low[:, 0] = np.arange(count, dtype=np.uint64)
    return O.to_mont(np.concatenate([top, low]))


@pytest.mark.parametrize("u", [1 << 16, (1 << 16) + 1])
def test_lookup_batch_edges(h2v, u):
    """One batch holding every edge of the batched scans and sorts at once, at u = 2^16 (n_pad == u: no padding keys) and
    u = 2^16 + 1 (n_pad = 2^17: almost half of every sorted slice is padding):
    a constant input (u - 1 repeated rows: the most leftover table values); an input of u distinct values (no repeated
    rows: rep_rows holds nothing for it and lookup_emit_table_batch_kernel finds no free table row); two lookups whose
    seam in the concatenated scans holds one value twice (the last sorted row of one and the first of the next are both
    1000: a first occurrence must not be judged across lookups); full-width values that differ only in the top or only
    in the lowest 32-bit limb (key_less); and an ordinary range lookup.  At 2^16 the distinct input is the last lookup
    (leftover count from totals is 0), at 2^16 + 1 the constant one is.  test_gpu_permute_batch_matches_per_lookup_oracle
    holds small-valued inputs of at most 5000 rows."""
    rng = np.random.default_rng(u)
    wide = _wide_families(rng, 40)
    seam_a = rng.integers(0, 1000, u, dtype=np.uint64)
    seam_a[rng.integers(u)] = 1000
    seam_b = rng.integers(1001, 2000, u, dtype=np.uint64)
    seam_b[rng.integers(u)] = 1000
    cases = {
        "range": (_mont(rng.integers(0, 1 << KMEANS_BITS, u, dtype=np.uint64)), 0),
        "seam_a": (_mont(seam_a), 0),
        "seam_b": (_mont(seam_b), 0),
        "constant": (_mont(np.full(u, 77, dtype=np.uint64)), 0),
        "distinct": (_mont(rng.permutation(u).astype(np.uint64)), 1),
        "wide": (wide[rng.integers(0, len(wide), u)], 2),
    }
    wide_table = np.concatenate([wide, O.fr_fill(u - len(wide), u + 7)])
    tables = [_range_table(KMEANS_BITS, u), _mont(rng.permutation(u).astype(np.uint64)), wide_table[rng.permutation(u)]]
    order = (["range", "seam_a", "seam_b", "wide", "constant", "distinct"] if u == 1 << 16 else
             ["distinct", "seam_a", "seam_b", "wide", "range", "constant"])
    lk = _Lookups(h2v, [cases[c][0] for c in order], tables, [cases[c][1] for c in order], u + 5)
    try:
        lk.run()
        lk.check(f"u = {u}, lookups {order}:")
    finally:
        lk.free()
