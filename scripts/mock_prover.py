"""Wall-clock time of h2v_mock_prover (MockProver::run on the device) and of h2v_pk_mock_prover (the same checks on a loaded
proving key, for a batch of witnesses) on the three reference examples (distances and query at k = 13, kmeans at k = 16)
and, with --sift, on the SIFT-shaped k = 20 circuit of scripts/sift_k20_proof.py.

    python scripts/mock_prover.py [--names distances query kmeans] [--reps 3] [--sift] [--out profiles/pk_mock_prover_b200.json]

The columns come from the restated builder and layouter (host numpy arrays, pageable).  Each circuit is checked once as a
warm-up, then `reps` times; the library reports each call's upload of the columns and its checks separately
(h2v_mock_last_ms).  query runs on data/query.in as it is, whose repeated vectors leave 12 gates unsatisfied, so its
number includes the compaction of real failures.  Then the circuit's proving key is loaded and checked with the key path:
its first call (which builds the key tables), then `reps` later calls with B = 1 and with B = 8 copies of the witness;
each witness's total must equal h2v_mock_prover's.  Writes one JSON object (also printed) with the GPU's name and power
limit read in the same run."""
import argparse
import json
import os
import random
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, limit = [x.strip() for x in out[0].split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:  # the numbers are still the GPU's: say that its limit could not be read
        return {"gpu": None, "power_limit": None, "nvidia_smi_error": str(e)}


def measure(h, rc, reps):
    cells = lambda cols: sum(int(c.shape[0]) for c in cols)
    run = lambda: h.MockProver.run(rc.cs, rc.fixed, rc.sigma, rc.advice, rc.instances)
    run()
    ups, chk, walls = [], [], []
    for _ in range(reps):
        t0 = time.perf_counter()
        mp = run()
        walls.append((time.perf_counter() - t0) * 1e3)
        ups.append(mp.upload_ms)
        chk.append(mp.check_ms)
    col_bytes = 32 * (cells(rc.advice) + cells(rc.fixed) + cells(rc.sigma))
    return {"k": rc.k, "advice_columns": len(rc.advice), "fixed_columns": len(rc.fixed), "permutation_columns": len(rc.cs["permutation"]),
            "gates": len(rc.cs["gates"]), "lookups": len(rc.cs["lookups"]), "column_gb": round(col_bytes / 1e9, 3),
            "n_failures": mp.n_failures, "upload_ms": [round(x, 2) for x in ups], "check_ms": [round(x, 2) for x in chk],
            "call_ms": [round(x, 2) for x in walls], "upload_gb_per_s": round(col_bytes / 1e6 / min(ups), 2)}


def measure_key(h, rc, reps, n_failures):
    """h2v_pk_mock_prover on the circuit's proving key: the first call, then later calls at B = 1 and B = 8"""
    srs = h.ParamsKZG.gen_srs(rc.k)
    t0 = time.perf_counter()
    pk = h.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, np.array([rc.k, 0, 0, 0], dtype=np.uint64))
    load_ms = (time.perf_counter() - t0) * 1e3

    def call(B):
        t0 = time.perf_counter()
        mps = pk.mock_prover([rc.advice] * B, [rc.instances] * B)
        wall = (time.perf_counter() - t0) * 1e3
        assert [m.n_failures for m in mps] == [n_failures] * B, [m.n_failures for m in mps]
        return {"upload_ms": round(mps[0].upload_ms, 2), "check_ms": round(mps[0].check_ms, 2), "call_ms": round(wall, 2)}

    out = {"pk_load_ms": round(load_ms, 1), "first_call_b1": call(1)}
    for B in (1, 8):
        runs = [call(B) for _ in range(reps)]
        out[f"later_b{B}"] = {key: [r[key] for r in runs] for key in runs[0]}
    pk.close()
    srs.close()
    return out


def measure_both(h, rc, reps):
    res = measure(h, rc, reps)
    res["pk_mock_prover"] = measure_key(h, rc, reps, res["n_failures"])
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--names", nargs="+", default=["distances", "query", "kmeans"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sift", action="store_true", help="also the k = 20 circuit of scripts/sift_k20_proof.py (1024 x 128)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pk_mock_prover_b200.json"))
    args = ap.parse_args()

    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import circuit as Z

    if h.device_count() < 1:
        raise SystemExit("mock_prover.py measures on a GPU; none is visible")
    h.init(0)
    res = {"what": "h2v_mock_prover wall-clock: upload of the columns and the checks, ms per call; pk_mock_prover: the same for "
                   "h2v_pk_mock_prover on the loaded key (first call with the key tables, later calls at B = 1 and 8 witnesses)",
           **gpu_info(), "circuits": {}}
    for name in args.names:
        k, bits = Z.EXAMPLE_PARAMS[name]
        rc, _ = Z.create_circuit(Z.EXAMPLES[name], Z.example_input(name), k, bits)
        res["circuits"][f"{name}_k{k}"] = measure_both(h, rc, args.reps)
        print(f"# {name}: {res['circuits'][f'{name}_k{k}']}", file=sys.stderr, flush=True)
        rc.close()
    if args.sift:
        # the circuit of scripts/sift_k20_proof.py: nearest_vector + merkle_commitment over 1024 random 128-dim vectors
        vectors, dim, k, bits = 1024, 128, 20, 19
        rnd = random.Random(20)
        inp = dict(query=[rnd.uniform(0.0, 2.0) for _ in range(dim)],
                   database=[[rnd.uniform(0.0, 2.0) for _ in range(dim)] for _ in range(vectors)])
        os.environ.setdefault("H2V_TRACE_RESERVE", str(int(vectors * dim * 2200)))
        builder = Z.GateThreadBuilder(bits)
        public = []
        Z.exhaustive_merkle(builder.main(0), inp, public)
        builder.make_public(public)
        rc = Z.RangeCircuit(builder, k)
        res["circuits"][f"sift_k{k}"] = measure_both(h, rc, min(args.reps, 2))
        print(f"# sift: {res['circuits'][f'sift_k{k}']}", file=sys.stderr, flush=True)
        rc.close()
        builder.close()
    res.update(gpu_info())          # read again after the run: the limit the measurement ran under
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f)
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
