"""Proofs per second of h2v_create_proofs (B proofs on one key in one call, run in groups phase by phase) against B
h2v_create_proof calls in a loop, on the three reference examples (distances and query at k = 13, kmeans at k = 16).

    python scripts/batch_prove.py [--names distances query kmeans] [--batches 1 2 4 8 16] [--rounds 3]

The columns come from the restated builder and layouter as bench.py's real_flow section builds them (advice in pinned
host memory).  For every B: one warm-up of each, then `rounds` alternations of the batch call and the loop, each with the
same B distinct seeds; every round checks that the batch's bytes equal the loop's.  An example stops growing B once a
batch no longer fits in one group (kmeans: about 12 GB of workspace per proof).  Prints one JSON line: per example
and B, proofs per second of each (best round), the groups the batch ran in, the batch's per-phase wall-clock
(h2v_pk_last_phase_ms, summed over its groups), and the GPU's name and power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--names", nargs="+", default=["distances", "query", "kmeans"])
    ap.add_argument("--batches", nargs="+", type=int, default=[1, 2, 4, 8, 16])
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import numpy as np
    import torch

    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import circuit as Z

    if not torch.cuda.is_available():
        raise SystemExit("batch_prove.py measures on a GPU; none is visible")
    h.init(0)
    L = h.lib()
    res = {"what": "proofs per second, h2v_create_proofs vs B h2v_create_proof calls", **gpu_info(),
           "torch_device": torch.cuda.get_device_name(0), "examples": {}}
    for name in args.names:
        k, bits = Z.EXAMPLE_PARAMS[name]
        n = 1 << k
        inp = Z.example_input(name)
        if name == "query":      # break the five-way ties of data/query.in (tests/test_circuit.py::test_query_layout)
            inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
        builder = Z.GateThreadBuilder(bits)
        public = []
        Z.EXAMPLES[name](builder.main(0), inp, public)
        builder.make_public(public)
        rc = Z.RangeCircuit(builder, k)
        srs = h.ParamsKZG.gen_srs(k)
        pk = h.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, np.array([k, 0, 0, 0], dtype=np.uint64))
        A = len(rc.advice)
        pinned = torch.empty((A, n, 4), dtype=torch.int64).pin_memory()
        adv = pinned.numpy().view(np.uint64)
        for i, c in enumerate(rc.advice):
            adv[i] = c
        cols = [adv[i] for i in range(A)]
        out = {}
        for B in args.batches:
            seeds = [bytes((p * 37 + j) % 256 for j in range(32)) for p in range(B)]
            batch = lambda: pk.create_proofs([cols] * B, [rc.instances] * B, seeds)
            loop = lambda: [pk.create_proof(cols, rc.instances, s) for s in seeds]
            batch()
            loop()
            tb, tl, phases, groups = [], [], None, None
            for _ in range(args.rounds):
                t0 = time.perf_counter()
                got = batch()
                tb.append(time.perf_counter() - t0)
                ph = (C.c_double * 8)()
                L.h2v_pk_last_phase_ms(pk._h, ph)
                phases, groups = pk.last_phase_ms(), int(ph[7])
                t0 = time.perf_counter()
                want = loop()
                tl.append(time.perf_counter() - t0)
                assert got == want, f"{name} B={B}: batch bytes differ from the single proofs"
            out[f"B{B}"] = {"batch_proofs_per_s": round(B / min(tb), 2), "loop_proofs_per_s": round(B / min(tl), 2),
                            "speedup": round(min(tl) / min(tb), 3), "batch_s": [round(t, 4) for t in tb], "loop_s": [round(t, 4) for t in tl],
                            "groups": groups, "group_size": -(-B // groups) if groups else None,
                            "batch_phase_ms": {kk: round(v, 2) for kk, v in phases.items()}}
            print(f"# {name} B={B}: {out[f'B{B}']}", file=sys.stderr, flush=True)
            if groups > 1:      # B is past the group size that fits: larger B only adds groups
                break
        res["examples"][f"{name}_k{k}"] = {"advice_columns": A, "lookups": len(rc.cs["lookups"]), "proof_bytes": pk.proof_size(), **out}
        pk.close()
        srs.close()
        del pinned, adv, cols
        rc.close()
        builder.close()
    res.update(gpu_info())          # read again after the run: the limit the measurement ran under
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
