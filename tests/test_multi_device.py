"""In-process multi-GPU (h2v_init(devices, n_dev), SURVEY.md 8(b) / 8(e)): handles hold one replica per device, the
host-facing batch entry points split their columns across the devices (column j -> device j mod G) and return results
in column order, `_dev` entry points run where their buffers live.  Needs >= 2 GPUs (skipped otherwise)."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture()
def two_devices(h2v):
    if h2v.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    h2v.init([0, 1])
    assert h2v.device_list() == [0, 1]
    yield h2v
    h2v.init(0)


def test_commit_batch_split_over_devices(two_devices):
    h = two_devices
    k, n = 10, 1 << 10
    bases = O.gen_bases(n)
    srs = h.ParamsKZG(k, None, bases)
    cols = [O.fr_fill(n, 300 + i, mode=i % 2) for i in range(11)]
    got = srs.commit_batch(cols)
    for g, c in zip(got, cols):
        assert (g == O.best_multiexp_affine(c, bases)).all()
    # single commits and short batches stay on the primary device
    assert (srs.commit_lagrange(cols[3]) == got[3]).all()
    srs.close()


def test_transform_batch_split_over_devices(two_devices):
    h = two_devices
    k = 9
    d, od = h.EvaluationDomain(4, k), O.EvaluationDomain(4, k)
    cols = [O.fr_fill(1 << k, 40 + i) for i in range(9)]
    for op, ref in ((h.OP_LAGRANGE_TO_COEFF, od.lagrange_to_coeff), (h.OP_COEFF_TO_EXTENDED, od.coeff_to_extended)):
        got = d.transform_batch(op, cols)
        for g, c in zip(got, cols):
            assert (g == ref(c)).all()
    d.close()


def test_dev_entry_points_run_where_the_buffers_live(two_devices):
    h = two_devices
    k, n = 9, 1 << 9
    bases = O.gen_bases(n)
    srs = h.ParamsKZG(k, None, bases)
    dom, od = h.EvaluationDomain(4, k), O.EvaluationDomain(4, k)
    cols = np.stack([O.fr_fill(n, 70 + i) for i in range(3)])
    for device in (0, 1):
        d_in = h.DeviceBuffer(cols.nbytes, device=device)
        d_in.upload(cols)
        d_out = h.DeviceBuffer(3 * 64, device=device)
        srs.commit_batch_dev(d_in.ptr, n, 3, n, d_out.ptr)
        got = d_out.download((3, 8))
        for i in range(3):
            assert (got[i] == O.best_multiexp_affine(cols[i], bases)).all(), (device, i)
        d_c = h.DeviceBuffer(cols.nbytes, device=device)
        dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_in.ptr, n, d_c.ptr, n, 3)
        coef = d_c.download((3, n, 4))
        for i in range(3):
            assert (coef[i] == od.lagrange_to_coeff(cols[i])).all(), (device, i)
    srs.close()
    dom.close()


def test_calls_return_on_the_device_they_were_addressed_to(two_devices):
    """an entry point leaves the calling thread's current device on the device its call was addressed to: the owner of
    its buffers, also when a resident batch was split over both devices, and the primary device for host columns"""
    import torch
    h = two_devices
    k, n, ncols = 9, 1 << 9, 21      # enough columns for both resident batches to be split
    torch.cuda.init()
    srs = h.ParamsKZG(k, None, O.gen_bases(n))
    dom = h.EvaluationDomain(4, k)
    cols = np.stack([O.fr_fill(n, 40 + i) for i in range(ncols)])
    d_in = h.DeviceBuffer(cols.nbytes, device=1)
    d_in.upload(cols)
    d_pts = h.DeviceBuffer(ncols * 64, device=1)
    d_c = h.DeviceBuffer(cols.nbytes, device=1)
    srs.commit_batch_dev(d_in.ptr, n, ncols, n, d_pts.ptr)
    assert torch.cuda.current_device() == 1
    for host_call in (lambda: h.batch_invert(cols[0]), lambda: h.g1_sum(np.zeros((0, 8), dtype=np.uint64))):
        dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_in.ptr, n, d_c.ptr, n, ncols)
        assert torch.cuda.current_device() == 1
        host_call()
        assert torch.cuda.current_device() == 0
    srs.close()
    dom.close()


def test_init_rejects_bad_lists(h2v):
    with pytest.raises(ValueError):
        h2v.init([0, 0])
    with pytest.raises(ValueError):
        h2v.init([h2v.device_count()])
    h2v.init(0)


def test_commit_batch_dev_split_over_devices(two_devices):
    """a resident batch of a proof phase: the columns are cut into one block per device, the other device pulls its block
    over NVLink and the results land in the owner's array in column order"""
    h = two_devices
    k, n = 9, 1 << 9
    bases = O.gen_bases(n)
    srs = h.ParamsKZG(k, None, bases)
    ncols = 37
    cols = np.stack([O.fr_fill(n, 500 + i, mode=i % 2) for i in range(ncols)])
    want = [O.best_multiexp_affine(cols[i], bases) for i in range(ncols)]
    for device in (0, 1):
        # contiguous columns (one peer copy) and columns with a gap between them (one copy per column)
        for stride in (n, n + 16):
            padded = np.zeros((ncols, stride, 4), dtype=np.uint64)
            padded[:, :n] = cols
            d_in = h.DeviceBuffer(padded.nbytes, device=device)
            d_in.upload(padded)
            d_out = h.DeviceBuffer(ncols * 64, device=device)
            srs.commit_batch_dev(d_in.ptr, stride, ncols, n, d_out.ptr)
            got = d_out.download((ncols, 8))
            for i in range(ncols):
                assert (got[i] == want[i]).all(), (device, stride, i)
    srs.close()


def test_transform_dev_split_over_devices(two_devices):
    h = two_devices
    k, n = 9, 1 << 9
    dom, od = h.EvaluationDomain(4, k), O.EvaluationDomain(4, k)
    ncols = 21
    cols = np.stack([O.fr_fill(n, 900 + i) for i in range(ncols)])
    for device in (0, 1):
        d_in = h.DeviceBuffer(cols.nbytes, device=device)
        d_in.upload(cols)
        d_c = h.DeviceBuffer(cols.nbytes, device=device)
        dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_in.ptr, n, d_c.ptr, n, ncols)
        coef = d_c.download((ncols, n, 4))
        d_e = h.DeviceBuffer(4 * cols.nbytes, device=device)
        dom.transform_dev(h.OP_COEFF_TO_EXTENDED, d_c.ptr, n, d_e.ptr, 4 * n, ncols)
        ext = d_e.download((ncols, 4 * n, 4))
        d_b = h.DeviceBuffer(4 * cols.nbytes, device=device)
        dom.transform_dev(h.OP_EXTENDED_TO_COEFF, d_e.ptr, 4 * n, d_b.ptr, 4 * n, ncols)
        back = d_b.download((ncols, 4 * n, 4))
        for i in range(ncols):
            c = od.lagrange_to_coeff(cols[i])
            assert (coef[i] == c).all(), (device, i)
            assert (ext[i] == od.coeff_to_extended(c)).all(), (device, i)
            assert (back[i][:n] == c).all() and not back[i][n:3 * n].any(), (device, i)
    dom.close()


def test_proof_bytes_do_not_depend_on_the_device_count(h2v):
    """create_proof with the commit phases spread over two devices: the same bytes as on one device and as the oracle's"""
    if h2v.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from common import fr_arr
    from oracle import plonk as PL
    from toy_circuit import Toy

    k, seed, secret = 8, bytes(range(32)), 0x1CE1CEBABE5EED0123456789ABCDEF0FEDCBA9876543210
    t = Toy(k, seed=5, n_gate_cols=22, n_lookup_cols=3)
    params = PL.Params.setup(k, secret)
    proofs = []
    for devs in ([0], [0, 1]):
        h2v.init(devs)
        srs = h2v.ParamsKZG(k, params.g, params.g_lagrange)
        pk = h2v.ProvingKey(srs, t.cs, [fr_arr(c) for c in t.fixed], [fr_arr(c) for c in t.sigma], fr_arr([t.vk_repr])[0])
        proofs.append(pk.create_proof([fr_arr(c) for c in t.advice], [fr_arr(c) for c in t.instances], seed))
        pk.close()
        srs.close()
    h2v.init(0)
    assert proofs[0] == proofs[1]
    assert proofs[0] == PL.create_proof(params, t.cs, t.fixed, t.sigma, t.vk_repr, t.advice, t.instances, seed)


@pytest.mark.parametrize("devices,k,cols_n", [pytest.param(1, 9, 19, id="1"), pytest.param(2, 9, 19, id="2"),
                                              pytest.param(4, 9, 37, id="4"), pytest.param(8, 9, 70, id="8"),
                                              pytest.param(1, 16, 40, id="1-k16")])
def test_commit_batch_resident(h2v, devices, k, cols_n):
    """h2v_commit_batch_resident: host columns are blinded, committed and left on the device (the advice phase of
    create_proof); with several devices each uploads and commits a block and forwards it to the owner.  At k = 16 the 40
    columns go up in two sub-batches of 32 and 8 (a full one holds 64 MiB of columns): the second crosses while the
    first is committed."""
    import torch
    if h2v.device_count() < devices:
        pytest.skip(f"needs {devices} GPUs")
    h2v.init(list(range(devices)) if devices > 1 else 0)
    try:
        n, rows = 1 << k, 6
        bases = O.gen_bases(n)
        srs = h2v.ParamsKZG(k, None, bases)
        cols = [O.fr_fill(n, 700 + i, mode=i % 2) for i in range(cols_n)]
        tails = np.stack([O.fr_fill(rows, 900 + i) for i in range(cols_n)])
        stride = n + 8
        dst = torch.zeros((cols_n, stride, 4), dtype=torch.int64, device="cuda:0")
        got = srs.commit_batch_resident(cols, tails, n - rows, dst.data_ptr(), stride)
        torch.cuda.synchronize(0)
        res = dst.cpu().numpy().view(np.uint64)
        for j in range(cols_n):
            want = cols[j].copy()
            want[n - rows:] = tails[j]
            assert (res[j, :n] == want).all() and not res[j, n:].any(), j
            assert (got[j] == O.best_multiexp_affine(want, bases)).all(), j
        srs.close()
    finally:
        h2v.init(0)
