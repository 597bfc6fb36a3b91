"""Child process of test_proof_size_parity.test_ntt_knobs_change_the_schedule_not_the_result.

The NTT schedule knobs (H2V_NTT_LOGE, H2V_NTT_SHOUP_MAX_L) are read once per process, so each setting needs a process
of its own.  This script runs under whatever environment its parent gave it: it reads `inputs.npz` from the directory
named on the command line, runs best_fft and the EvaluationDomain ops on cuda:0 and writes every result to
`outputs.npz` in the same directory, for the parent to compare with the oracle.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import halo2_vectordb_b200 as h  # noqa: E402


def main(work):
    h.init(0)
    inp = np.load(os.path.join(work, "inputs.npz"))
    out = {}
    for key in inp.files:
        if key.startswith("fft_a_"):
            log_n = int(key[len("fft_a_"):])
            out[f"fft_{log_n}"] = h.best_fft(inp[key], inp[f"fft_w_{log_n}"], log_n)
        elif key.startswith("dom_a_"):
            k = int(key[len("dom_a_"):])
            d = h.EvaluationDomain(4, k)
            a, e = inp[key], inp[f"dom_e_{k}"]
            out[f"l2c_{k}"] = d.lagrange_to_coeff(a)
            out[f"c2l_{k}"] = d.coeff_to_lagrange(a)
            out[f"c2e_{k}"] = d.coeff_to_extended(a)
            out[f"e2c_{k}"] = d.extended_to_coeff(e)
            out[f"dvp_{k}"] = d.divide_by_vanishing_poly(e)
            out[f"fused_{k}"] = d.transform_batch(h.OP_DIVIDE_BY_VANISHING, [e])[0]
            d.close()
    np.savez(os.path.join(work, "outputs.npz"), **out)


if __name__ == "__main__":
    main(sys.argv[1])
