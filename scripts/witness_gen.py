"""Witness generation on the GPU (WitnessProgram.generate, h2v_witness_generate) against the host builder + RangeCircuit,
on the reference examples (distances and query at k = 13, kmeans at k = 16) and, with --sift, the SIFT-shaped query
(nearest_vector + merkle_commitment over 1024 x 128 at k = 20).

    python scripts/witness_gen.py [--names distances query kmeans] [--batches 1 8 32] [--sift]

For every example: one recording, one program; then for every B, B distinct inputs (the recording's, shifted by w / 64)
are generated in one call (after a warm-up call) and built on the host one by one, and every generated witness is
checked byte for byte against the host's.  Then inputs -> proofs three ways, each over all B witnesses in chunks of 8
with the same seeds: host builder + layout per witness then create_proofs; generate then create_proofs; and
create_proofs_from_inputs, which generates the columns in the key's workspace (no columns on the host).  The proofs of
the three flows must be equal.  Prints one JSON line: per example and B the host and GPU seconds per witness, the
program's levels, cells and folded share, generate's upload / evaluate / download ms, proofs per second of the three
flows, the new flow's phase-0 and generation ms, and the GPU's name and power limit read in the same run.  --out PATH
also rewrites that JSON to PATH after every line, so that a run that ends early keeps what it measured."""
import argparse
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


def shifted(inp, d):
    return {key: ([[x + d for x in v] for v in val] if isinstance(val[0], list) else [x + d for x in val]) for key, val in inp.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--names", nargs="+", default=["distances", "query", "kmeans"])
    ap.add_argument("--batches", nargs="+", type=int, default=[1, 8, 32])
    ap.add_argument("--sift", action="store_true")
    ap.add_argument("--no-proofs", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import random

    import numpy as np

    import halo2_vectordb_b200 as h
    from halo2_vectordb_b200 import circuit as Z

    if h.lib().h2v_device_count() < 1:
        raise SystemExit("witness_gen.py measures on a GPU; none is visible")
    h.init(0)
    res = {"what": "witness generation: host builder + RangeCircuit vs WitnessProgram.generate; inputs -> proofs three ways",
           "command": f"scripts/witness_gen.py --names {' '.join(args.names)} --batches {' '.join(map(str, args.batches))}"
                      + (" --sift" if args.sift else "") + (" --no-proofs" if args.no_proofs else ""), **gpu_info(), "examples": {}}
    cases = [(name, Z.EXAMPLES[name], Z.example_input(name), *Z.EXAMPLE_PARAMS[name]) for name in args.names]
    if args.sift:
        rnd = random.Random(20)
        inp = dict(query=[rnd.uniform(0.0, 2.0) for _ in range(128)], database=[[rnd.uniform(0.0, 2.0) for _ in range(128)] for _ in range(1024)])
        cases.append(("sift", Z.exhaustive_merkle, inp, 20, 19))
    for name, f, inp, k, bits in cases:
        if name == "query":      # break the five-way ties of data/query.in, so that every witness satisfies the circuit
            inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
        t0 = time.perf_counter()
        rec = Z.create_circuit(f, inp, k, bits, record=True)[0]
        t_rec = time.perf_counter() - t0
        t0 = time.perf_counter()
        prog = Z.WitnessProgram(rec.builder, k)
        t_prog = time.perf_counter() - t0
        info = prog.info
        quant = Z.FixedPointChip.default(rec.builder)

        def leaves(x):
            if name == "sift":
                return quant.quantize_vector(list(x["query"]) + [v for row in x["database"] for v in row])
            return Z.example_witness_inputs(name, x)

        ex = {"k": k, "record_s": round(t_rec, 3), "program_s": round(t_prog, 3), "levels": info["levels"], "cells": info["cells"],
              "computed_cells": info["computed_cells"], "folded_share": round(1 - info["computed_cells"] / info["cells"], 4),
              "bytes_per_witness": info["bytes_per_witness"], "batches": {}}
        srs = pk = None
        if not args.no_proofs:
            srs = h.ParamsKZG.gen_srs(k)
            pk = h.ProvingKey(srs, rec.cs, rec.fixed, rec.sigma, np.array([k, 0, 0, 0], dtype=np.uint64))
        for B in args.batches:
            ins = [shifted(inp, w / 64) for w in range(B)]
            x = [leaves(v) for v in ins]
            prog.generate(x[:1])      # warm-up
            t0 = time.perf_counter()
            gen = prog.generate(x)
            t_gen = time.perf_counter() - t0
            ms = prog.last_ms()
            t_host, same = 0.0, True
            for (adv, inst), v in zip(gen, ins):      # one host layout at a time: a kmeans layout holds 2.3 GB
                t0 = time.perf_counter()
                rc = Z.create_circuit(f, v, k, bits)[0]
                t_host += time.perf_counter() - t0
                same &= all(a.tobytes() == b.tobytes() for a, b in zip(adv, rc.advice)) and inst[0].tobytes() == rc.instances[0].tobytes()
                rc.close()
            del gen
            row = {"host_s_per_witness": round(t_host / B, 5), "generate_s_per_witness": round(t_gen / B, 5),
                   "generate_ms": {"upload": round(ms[0], 3), "evaluate_gather": round(ms[1], 3), "download": round(ms[2], 3)},
                   "bytes_equal": same}
            if pk is not None:      # inputs -> proofs, each flow in chunks of at most 8 witnesses (host memory)
                seeds = [bytes([w % 256]) * 32 for w in range(B)]
                chunks = [(ins[c0:c0 + 8], seeds[c0:c0 + 8]) for c0 in range(0, B, 8)]
                p_host, p_gen, p_dev, t_host_e2e, t_gen_e2e, t_dev_e2e, phase0, wms = [], [], [], 0.0, 0.0, 0.0, 0.0, [0.0] * 3
                for chunk, sd in chunks:
                    t0 = time.perf_counter()
                    hs = [Z.create_circuit(f, v, k, bits)[0] for v in chunk]
                    p_host += pk.create_proofs([rc.advice for rc in hs], [rc.instances for rc in hs], sd)
                    t_host_e2e += time.perf_counter() - t0
                    del hs
                for chunk, sd in chunks:
                    t0 = time.perf_counter()
                    g = prog.generate([leaves(v) for v in chunk])
                    p_gen += pk.create_proofs([a for a, _ in g], [i for _, i in g], sd)
                    t_gen_e2e += time.perf_counter() - t0
                    del g
                for chunk, sd in chunks:
                    t0 = time.perf_counter()
                    p_dev += pk.create_proofs_from_inputs(prog, [leaves(v) for v in chunk], sd)[0]
                    t_dev_e2e += time.perf_counter() - t0
                    phase0 += pk.last_phase_ms()["advice_commit"]
                    wms = [a + b for a, b in zip(wms, prog.last_ms())]
                row.update(proofs_per_s_host=round(B / t_host_e2e, 3), proofs_per_s_generate=round(B / t_gen_e2e, 3),
                           proofs_per_s_from_inputs=round(B / t_dev_e2e, 3), from_inputs_phase0_ms=round(phase0, 3),
                           from_inputs_generate_ms={"upload": round(wms[0], 3), "evaluate_gather": round(wms[1], 3),
                                                    "instances_download": round(wms[2], 3)},
                           proofs_equal=p_host == p_gen == p_dev)
            ex["batches"][str(B)] = row
            res["examples"][name] = ex
            print(json.dumps({name: {str(B): row}}), file=sys.stderr, flush=True)
            if args.out:
                with open(args.out, "w") as fo:
                    json.dump(res, fo, indent=1)
        if pk is not None:
            pk.close()
            srs.close()
        prog.close()
        res["examples"][name] = ex
    print(json.dumps(res))


if __name__ == "__main__":
    main()
