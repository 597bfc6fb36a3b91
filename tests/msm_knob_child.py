"""Child process of test_proof_shape_batches.test_msm_knobs_change_the_schedule_not_the_result.

The MSM knobs (H2V_SCATTER_SLICES, H2V_RED_WEIGHT, H2V_CHUNK) are read once per process, so each setting needs a
process of its own.  This script runs under whatever environment its parent gave it: it reads `inputs.npz` from the
directory named on the command line (`cols_16`: columns of 2^16 scalars, `cols_20`: columns of 2^20 scalars), commits
them device-resident against ParamsKZG(16) / ParamsKZG(20) on the synthetic bases on cuda:0 -- all columns of a size in
one commit_batch_dev call, and column 1 of `cols_20` alone -- and writes the commitments and the (window bits, windows)
of each SRS's main table to `outputs.npz` in `out_dir`, for the parent to compare with the oracle.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import halo2_vectordb_b200 as h  # noqa: E402


def commit_dev(srs, cols):
    count, n = cols.shape[0], cols.shape[1]
    d_cols, d_out = h.DeviceBuffer(cols.nbytes), h.DeviceBuffer(count * 64)
    d_cols.upload(cols)
    srs.commit_batch_dev(d_cols.ptr, n, count, n, d_out.ptr)
    got = d_out.download((count, 8))
    d_cols.free()
    d_out.free()
    return got


def main(work, out_dir):
    h.init(0)
    out = {}
    with np.load(os.path.join(work, "inputs.npz")) as inp:
        for k in (16, 20):
            cols = inp[f"cols_{k}"]
            srs = h.ParamsKZG(k, None, h.synthetic_bases(1 << k))
            out[f"window_{k}"] = np.array(srs.info(), dtype=np.uint32)      # before any commit: the main table
            out[f"commit_{k}"] = commit_dev(srs, cols)
            if k == 20:
                out["commit_20_one"] = commit_dev(srs, cols[1:2])
            srs.close()
    np.savez(os.path.join(out_dir, "outputs.npz"), **out)


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
