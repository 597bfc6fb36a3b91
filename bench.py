#!/usr/bin/env python
"""bench.py -- the KZG-commit / EvaluationDomain hot path on N B200s (one process per GPU).

Workload (BASELINE.json configs[2], the 20x target): the kmeans circuit at k = 16.  One *step* is one
pass of the hot path over one batch of synthetic columns: `commit_lagrange` (BN254 G1 MSM against the
shared g_lagrange bases) of COLS columns of n = 2^16 Fr scalars.  The headline metric is
G1 MSM throughput in Mpts/s (BASELINE.json: "G1 MSM Mpts/s"); the same JSON line also carries the Fr
NTT throughput (Gelem/s) and a prove-shaped latency for the same circuit under "ntt" / "prove_shaped".

  value   device-resident: columns already in HBM when the timed region starts
  e2e     through the host-facing C ABI (h2v_commit_batch) with pinned HOST buffers: H2D of every
          column and D2H of every commitment inside the timed region
  roofline  dominant kernel msm_accumulate against the integer pipe (measured IMAD.WIDE peak), per
          SURVEY.md 8(d); "ntt.roofline" carries the HBM view for the NTT passes
  cpu_baseline / --impl reference   the restated halo2-axiom CPU path (oracle/, kind "port": the Rust
          reference cannot be built in this image) on all host cores, on a bounded sample

N > 1: columns are partitioned across ranks (each rank commits its own COLS columns against its own
SRS replica), no data-path collective; scaling = weak.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K = 16
N = 1 << K
COLS = 96                      # 96 x 2 MiB of scalars = 192 MiB per step (> 126 MB L2), tables 64 MiB more
MSM_MACS_PER_POINT = {16: 27200, 13: 27200, 20: 20400}   # SURVEY.md 8(d): W(n) * 1360 wide-MACs
FQ_MUL_MACS = 136
SHOUP_MUL_MACS = 107         # twiddle product of the NTT (csrc/shoup.cuh): 99 IMAD.WIDE + 16 low-only IMAD at half the pipe time
FQ_SQR_MACS = 108                 # the dedicated squaring: 28 + 8 products, 64 + 8 reduction
MIXED_ADD_MACS = 8 * FQ_MUL_MACS + 2 * FQ_SQR_MACS      # what msm_accumulate executes per sorted entry (SURVEY counts 10 x 136 = 1360)
ACC_DRAM_BYTES_PER_LAUNCH = 4.13e9   # msm_accumulate_kernel, 96 columns x 2^16, c = 15: 3.709 GB read + 0.421 GB written (ncu --set full, final build of round 2)
SYN_A, SYN_B = 0x9E3779B97F4A7C15 >> 2, 0x632BE59BD9B4E019 >> 2


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cols", type=int, default=COLS)
    ap.add_argument("--no-extras", action="store_true", help="skip the ntt / prove_shaped / cpu_baseline sections")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the commitments of the last timed step as DIR/<name>.npy (rank 0's columns), so that two "
                         "builds can be compared output for output; the inputs depend only on the arguments")
    return ap.parse_args()


def dump_outputs(path, points):
    """points: {name: (n, 8) G1Affine, 64-bit Montgomery limbs} -> DIR/<name>.npy, (n, 2, 8) float64: x and y as eight
    little-endian 32-bit limbs each, which float64 holds exactly"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, p in points.items():
        limbs = np.ascontiguousarray(p, dtype="<u8").view("<u4").reshape(len(p), 2, 8)
        np.save(os.path.join(path, name + ".npy"), limbs.astype(np.float64))


# ----------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                pass
        sm = [int(r[0]) for r in self.rows if len(r) >= 7 and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) >= 7 and r[1].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------- CPU arm
def cpu_msm_sample(n_cols, threads):
    """restated halo2-axiom best_multiexp on `n_cols` columns of 2^16 uniform scalars, all host threads"""
    from oracle import oracle as O
    bases = O.gen_bases(N, threads=threads)
    cols = [O.fr_fill(N, 7000 + i) for i in range(n_cols)]
    t = time.perf_counter()
    for c in cols:
        O.best_multiexp(c, bases, threads)
    dt = time.perf_counter() - t
    return n_cols * N / dt / 1e6, dt


def cpu_ntt_sample(threads):
    """restated halo2-axiom EvaluationDomain on the host cores: seconds per lagrange_to_coeff (2^16) and
    coeff_to_extended (2^16 -> 2^18)"""
    from oracle import oracle as O
    d = O.EvaluationDomain(4, K)
    a = O.fr_fill(N, 4321)
    d.lagrange_to_coeff(a, threads)
    t = time.perf_counter()
    for _ in range(4):
        d.lagrange_to_coeff(a, threads)
    t_l2c = (time.perf_counter() - t) / 4
    t = time.perf_counter()
    for _ in range(2):
        d.coeff_to_extended(a, threads)
    t_c2e = (time.perf_counter() - t) / 2
    return t_l2c, t_c2e


def run_reference(args, rank, world, out):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from oracle import oracle as O
    sample_cols = min(24, args.cols)      # a bounded sample of the step's 96 columns: the metric is a rate
    bases = O.gen_bases(N, threads=threads)
    cols = [O.fr_fill(N, 7000 + i) for i in range(sample_cols)]
    for _ in range(min(args.warmup, 1)):
        O.best_multiexp(cols[0], bases, threads)
    t = time.perf_counter()
    for _ in range(args.steps):
        last = [O.best_multiexp(c, bases, threads) for c in cols]
    dt = time.perf_counter() - t
    if args.dump_outputs:
        import numpy as np
        dump_outputs(args.dump_outputs, {"commitments": np.stack([O.g1_to_affine(p) for p in last])})
    v = args.steps * sample_cols * N / dt / 1e6
    sample = f"{sample_cols} columns of 2^16 uniform Fr per step (of the {args.cols}-column batch), best_multiexp over {threads} threads"
    print(file=out, *[json.dumps({
        "impl": "reference", "metric": "msm_mpts_per_s", "value": v, "unit": "Mpts/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "dtype_note": "4 x 64-bit limbs, Montgomery form (CPU restatement)", "data": "synthetic",
        "config": {"workload": "kmeans k=16 commit_lagrange batch (BASELINE configs[2])", "k": K, "cols_per_step": args.cols,
                   "scalars": "uniform", "sampled_cols_per_step": sample_cols, "parallelism": f"{threads} host threads"},
        "cpu_baseline": {"value": v, "unit": "Mpts/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mpts/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "restated halo2-axiom CPU path (oracle/bn254_oracle.c); the Rust reference cannot be built here (no cargo, un-vendored deps)",
    })])


# ----------------------------------------------------------------------------------- GPU arm
def main():
    args = parse()
    # rank 0 must print exactly ONE JSON line: park the real stdout and send everything else (NCCL's version
    # banner, library chatter) to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    try:
        _main(args, real_stdout)
    finally:
        real_stdout.flush()


def _main(args, real_stdout):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world, real_stdout)
        return

    import numpy as np
    import torch
    import halo2_vectordb_b200 as h

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        # the ranks that have no extras to run wait for rank 0 on the CPU: a NCCL barrier would park a spinning kernel on
        # their GPUs, which rank 0 drives itself in the in-process N-GPU proof (real_flow_n_gpus)
        cpu_group = dist.new_group(backend="gloo")
    h.init(local_rank)
    cols = args.cols

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- synthetic inputs: bases with known discrete logs (device-generated), uniform scalars
    bases = h.synthetic_bases(N, SYN_A, SYN_B)
    srs = h.ParamsKZG(K, None, bases)
    g = torch.Generator(device="cpu").manual_seed(1234 + rank)
    host = torch.randint(-(1 << 63), (1 << 63) - 1, (cols, N, 4), dtype=torch.int64, generator=g)
    host[..., 3] &= (1 << 60) - 1                      # any value < 2^252 < r is a valid Montgomery residue
    host = host.pin_memory()
    d_cols = host.to(dev)
    d_out = torch.zeros((cols, 8), dtype=torch.int64, device=dev)
    out_host = np.zeros((cols, 8), dtype=np.uint64)
    host_np = host.numpy().view(np.uint64)
    import ctypes as C
    col_ptrs = (C.c_void_p * cols)(*[host_np[i].ctypes.data for i in range(cols)])

    def step_dev():
        srs.commit_batch_dev(d_cols.data_ptr(), N, cols, N, d_out.data_ptr())

    def step_e2e():
        h._check(h.lib().h2v_commit_batch(srs._h, h.H2V_BASIS_LAGRANGE, col_ptrs, cols, N, out_host.ctypes.data_as(C.c_void_p)))

    # integer-pipe peak, measured live (MEASURED_PEAKS.json has none).  Three probes, none of which is a kernel under test:
    #   row    a loop of nothing but carry-chained IMAD.WIDE.U32.X rows on independent accumulators (h2v_selftest_imad_probe(1))
    #   chain  a register-resident Fq Montgomery-product chain x 136 wide-MACs per product (h2v_selftest_op_rate)
    #   r01    round 1's loop-variant mad.wide.u32 stream (its 64-bit accumulate splits into IMAD.WIDE + 2 IADD3: reads low)
    # The denominator is the highest rate the pipe demonstrably sustains; the nominal figure is 148 SM x 32 / clk.
    peak_row, peak_chain, peak_r01 = h.imad_probe(1), h.op_rate(1) * FQ_MUL_MACS, h.imad_peak()
    peak = max(peak_row, peak_chain, peak_r01)

    # ---- device-resident timing
    # the clock sampler starts before the warm-up (nvidia-smi needs a few hundred ms to deliver its first
    # line); warm-up and timed steps are the same load, so every sample is taken under load
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step_dev()
    kernel_ms = {k: 0.0 for k in h.KERNEL_CLASSES}
    barrier()
    l0 = h.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_dev()
        for kk, v in h.last_kernel_ms().items():
            kernel_ms[kk] += v
    e1.record()
    barrier()
    launches = h.launch_count() - l0
    clocks = sampler.stop()
    dt = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    value = world * args.steps * cols * N / dt / 1e6

    # correctness guard on the timed result: column 0 against the closed form, via the C ABI result
    got0 = d_out[0].cpu().numpy().view(np.uint64)

    # ---- end to end through the host-facing C ABI
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    barrier()
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    barrier()
    dt_e2e = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    e2e_value = world * args.steps * cols * N / dt_e2e / 1e6
    assert (out_host[0] == got0).all(), "device-resident and host-facing paths disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"commitments": d_out.cpu().numpy().view(np.uint64), "commitments_e2e": out_host})

    acc_ms = kernel_ms["msm_accumulate"] / args.steps           # one launch per step (all columns)
    macs = cols * N * MSM_MACS_PER_POINT[K]
    achieved = macs / (acc_ms * 1e-3) / 1e12 if acc_ms > 0 else None
    executed = (cols * N * srs.info()[1] * MIXED_ADD_MACS) / (acc_ms * 1e-3) / 1e12 if acc_ms > 0 else None
    line = {
        "metric": "msm_mpts_per_s", "value": value, "unit": "Mpts/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "dtype_note": "8 x 32-bit limbs, Montgomery form, BN254 Fq/Fr (IMAD.WIDE 32x32+64)", "data": "synthetic",
        "config": {"workload": "kmeans k=16 commit_lagrange batch (BASELINE configs[2])", "k": K, "cols_per_step": cols,
                   "scalars": "uniform", "l2": "inputs larger than L2 (192 MiB scalars + 64 MiB tables per step)",
                   "parallelism": f"columns x{world}"},
        "e2e": {"value": e2e_value, "unit": "Mpts/s", "h2d_bytes_per_step": cols * N * 32, "d2h_bytes_per_step": cols * 64,
                "ms_per_step": dt_e2e / args.steps * 1e3},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "kernel_ms_per_step": {k: round(v / args.steps, 4) for k, v in kernel_ms.items() if v},
        "roofline": {"bound": "int32-pipe (IMAD.WIDE)", "kernel": "msm_accumulate_kernel", "achieved": achieved,
                     "peak": peak / 1e12, "unit": "T wide-MAC/s",
                     # frac: the wide multiply-adds the kernel EXECUTES (17 signed windows x 1304 per point: 8 products + 2 dedicated squarings per mixed addition) over the measured peak;
                     # frac_algorithmic: SURVEY 8(d)'s count (20 unsigned windows) over the same peak -- above 1 because the
                     # precomputed-table layout needs fewer windows, not because the pipe runs faster than its peak
                     "frac": (executed / (peak / 1e12)) if executed else None,
                     "frac_algorithmic": (achieved / (peak / 1e12)) if achieved else None,
                     "executed": executed,
                     "traffic": ACC_DRAM_BYTES_PER_LAUNCH if cols == COLS else None,
                     "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full of this launch (profiles/r02_final2_ncu_summary.txt)",
                     "peak_probes": {"imad_wide_x_rows": peak_row / 1e12, "fq_product_chain_x136": peak_chain / 1e12,
                                     "r01_mad_wide_stream": peak_r01 / 1e12, "nominal_148sm_x_32_per_clk_at_1965mhz": 9.31},
                     "peak_source": "measured live, max of the probes (none of them is the kernel under test); MEASURED_PEAKS.json has no integer peak",
                     "window_bits": srs.info()[0], "windows": srs.info()[1],
                     "algorithmic": f"{MSM_MACS_PER_POINT[K]} wide-MAC/pt x {cols * N} pts per launch (SURVEY.md 8d)"},
    }

    # ---- strong scaling: ONE fixed commit phase of the kmeans k = 16 proof (1 150 columns of 2^16, SURVEY.md App. C) split
    # over the ranks by column index, host columns in, commitments gathered back in column order inside the timed region
    line["strong"] = bench_strong_phase(h, torch, dev, srs, host_np, rank, world, barrier, max_over_ranks)
    if not args.no_extras:
        # the same for BASELINE configs[3] (SIFT-shaped, k = 20: ~360 commits of 2^20 per proof, SURVEY.md App. C)
        try:
            n20 = 1 << 20
            from halo2_vectordb_b200.synthetic import uniform_scalars
            srs20 = h.ParamsKZG(20, None, h.synthetic_bases(n20, SYN_A, SYN_B))
            host20 = torch.from_numpy(uniform_scalars(8, n20, 20 + rank).view(np.int64)).pin_memory().numpy().view(np.uint64)
            line["strong_k20"] = bench_strong_phase(h, torch, dev, srs20, host20, rank, world, barrier, max_over_ranks, total_cols=STRONG_COLS_K20,
                                                    n=n20, what="one SIFT-shaped k=20 proof's commits")
            srs20.close()
            del host20
            torch.cuda.empty_cache()
        except Exception as e:      # never lose the headline line to an extra
            line["strong_k20"] = {"error": str(e)[:200]}

    if not args.no_extras and rank == 0:
        line["ntt"] = bench_ntt(h, torch, dev, peak)
        line["witness_like"] = bench_witness(h, torch, dev, srs, peak)
        line["prove_shaped"] = bench_prove_shaped(h, torch, dev, srs, d_cols, cols)
        if not os.environ.get("H2V_BENCH_SKIP_REAL"):
            rf = bench_real_flow(h, torch)
            line["prove_shaped"]["real_flow"] = rf
            line["prove_shaped"]["kmeans_k16_real_flow_s"] = rf["kmeans_k16"]["prove_s"]
            if world > 1 and not os.environ.get("H2V_BENCH_SKIP_MULTI"):
                # the same kmeans proof with the commit / transform batches of every phase spread over the job's N GPUs in
                # process (rank 0 drives all of them; the other ranks are idle at the final barrier)
                try:
                    line["prove_shaped"]["real_flow_n_gpus"] = bench_real_flow_multi(h, torch, world)
                except Exception as e:      # never lose the headline line to the extra
                    line["prove_shaped"]["real_flow_n_gpus"] = {"error": str(e)[:200]}
                h.init(local_rank)
        line["next_row2"] = bench_row2(h, torch, dev, d_cols, cols)
        line["next_row1"] = bench_row1(h, torch, dev)
        if world == 1:
            threads = os.cpu_count() or 1
            v, secs = cpu_msm_sample(24, threads)
            t_l2c, t_c2e = cpu_ntt_sample(threads)
            n_msm, n_intt, n_cntt = PROVE_SHAPES["kmeans_k16"][1:4]
            line["cpu_baseline"] = {"value": v, "unit": "Mpts/s", "cores": threads, "kind": "port",
                                    "ntt_ms": {"lagrange_to_coeff_2^16": t_l2c * 1e3, "coeff_to_extended_2^18": t_c2e * 1e3},
                                    "prove_shaped_kmeans_k16_s": n_msm * N / (v * 1e6) + n_intt * t_l2c + n_cntt * t_c2e,
                                    "prove_shaped_note": "extrapolated from the sampled per-call times with the same call counts as prove_shaped.kmeans_k16",
                                    "sample": f"24 of the {cols} columns (2^16 uniform Fr each), restated halo2-axiom best_multiexp, {secs:.1f} s"}
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier(group=cpu_group)
    if rank == 0:
        print(json.dumps(line), file=real_stdout)
    srs.close()
    if world > 1:
        dist.destroy_process_group()


STRONG_COLS = 1150     # commit_lagrange calls of one kmeans k = 16 proof (SURVEY.md App. C)
STRONG_COLS_K20 = 360  # ... of one SIFT-shaped k = 20 proof


def bench_strong_phase(h, torch, dev, srs, host_np, rank, world, barrier, max_over_ranks, total_cols=None, n=None, what=None):
    """One fixed phase split over the ranks (scaling = strong): column j of STRONG_COLS goes to rank j mod world; every rank
    commits its share through the host-facing entry point (pinned host columns, H2D inside), then the commitments are
    all-gathered and put back in column order -- what the host transcript of ONE proof needs before the next challenge.
    The same columns are reused round-robin from the step's pinned batch (the data does not matter for the timing of
    uniform scalars).  Timed as max over ranks, gather included."""
    import ctypes as C
    import numpy as np
    STRONG_COLS = total_cols or globals()["STRONG_COLS"]
    N = n or globals()["N"]
    mine = [j for j in range(STRONG_COLS) if j % world == rank]
    per = (STRONG_COLS + world - 1) // world
    ptrs = (C.c_void_p * len(mine))(*[host_np[j % host_np.shape[0]].ctypes.data for j in mine])
    out = np.zeros((per, 8), dtype=np.uint64)
    out_t = torch.from_numpy(out.view(np.int64))
    gathered = torch.zeros((world, per, 8), dtype=torch.int64, device=dev)
    ordered = torch.zeros((STRONG_COLS, 8), dtype=torch.int64)

    def phase():
        h._check(h.lib().h2v_commit_batch(srs._h, h.H2V_BASIS_LAGRANGE, ptrs, len(mine), N, out.ctypes.data_as(C.c_void_p)))
        if world > 1:
            import torch.distributed as dist
            dist.all_gather_into_tensor(gathered, out_t.to(dev))
            g = gathered.cpu()
        else:
            g = out_t.unsqueeze(0)
        for r in range(world):                       # rank r holds columns r, r + world, ...
            cnt = len(range(r, STRONG_COLS, world))
            ordered[r::world] = g[r, :cnt]
        return ordered

    phase()
    ts = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        phase()
        torch.cuda.synchronize()
        ts.append(max_over_ranks(time.perf_counter() - t0))
    t = min(ts)
    what = what or "one kmeans k=16 proof's commits"
    return {"scaling": "strong", "phase": f"commit_lagrange of {STRONG_COLS} columns x 2^{N.bit_length() - 1} ({what}), host columns in, "
                                          "commitments gathered in column order", "n_gpus": world, "ms": t * 1e3,
            "mpts_per_s": STRONG_COLS * N / t / 1e6, "cols_per_rank": len(mine)}


def bench_real_flow(h, torch, names=("distances", "query", "kmeans")):
    """ONE real proof per reference example (BASELINE configs[0..2]): the witness comes from the restated chips on the
    example's own input (halo2_vectordb_b200.circuit: /root/reference/examples/{distances,query,kmeans}.rs on
    data/*.in), the columns from the restated halo2-base layouter, and the proof from h2v_create_proof -- the seed-zero
    SRS of gen_srs, ChaCha20 blinding, the Poseidon transcript, real challenge dependencies between the phases, SHPLONK
    opening: every step of SURVEY.md 3.1 from the advice columns (pinned host memory) to the proof bytes.  `prove_s` is
    create_proof alone; the host-side witness generation and layout (serial upstream as well) are timed beside it."""
    import numpy as np
    from halo2_vectordb_b200 import circuit as Z
    res = {}
    for name in names:
        k, bits = Z.EXAMPLE_PARAMS[name]
        n = 1 << k
        inp = Z.example_input(name)
        if name == "query":      # break the five-way ties of data/query.in (tests/test_circuit.py::test_query_layout)
            inp["database"] = [[x + 1e-3 * (i // 4) for x in v] for i, v in enumerate(inp["database"])]
        t0 = time.perf_counter()
        builder = Z.GateThreadBuilder(bits)
        public = []
        Z.EXAMPLES[name](builder.main(0), inp, public)
        builder.make_public(public)
        t_wit = time.perf_counter() - t0
        st = builder.stats()
        t0 = time.perf_counter()
        rc = Z.RangeCircuit(builder, k)
        t_lay = time.perf_counter() - t0
        t0 = time.perf_counter()
        srs = h.ParamsKZG.gen_srs(k)
        t_srs = time.perf_counter() - t0
        t0 = time.perf_counter()
        vk_repr = np.array([k, 0, 0, 0], dtype=np.uint64)
        pk = h.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, vk_repr)
        t_pk = time.perf_counter() - t0
        A = len(rc.advice)
        pinned = torch.empty((A, n, 4), dtype=torch.int64).pin_memory()
        adv = pinned.numpy().view(np.uint64)
        for i, c in enumerate(rc.advice):
            adv[i] = c
        cols = [adv[i] for i in range(A)]
        proof = pk.create_proof(cols, rc.instances, bytes(32))
        ts, phases = [], None
        for _ in range(3):
            t0 = time.perf_counter()
            p2 = pk.create_proof(cols, rc.instances, bytes(32))
            ts.append(time.perf_counter() - t0)
            phases = pk.last_phase_ms()
            assert p2 == proof, "create_proof is not deterministic in the seed"
        res[f"{name}_k{k}"] = {
            "prove_s": min(ts), "k": k, "lookup_bits": bits, "advice_cells": st["advice_cells"], "lookup_cells": st["lookup_cells"],
            "advice_columns": rc.num_advice, "lookup_advice_columns": rc.num_lookup_advice, "fixed_columns": len(rc.fixed),
            "permutation_columns": len(rc.cs["permutation"]), "public_inputs": rc.num_instances, "proof_bytes": len(proof),
            "phase_ms": {kk: round(v, 2) for kk, v in phases.items()},
            "host_s": {"witness_generation": round(t_wit, 3), "layout_and_sigma": round(t_lay, 3)},
            "setup_s": {"gen_srs": round(t_srs, 2), "pk_load": round(t_pk, 2)}}
        pk.close()
        srs.close()
        del pinned, adv, cols
        rc.close()
        builder.close()
    res["note"] = ("one real create_proof per reference example: witness by the restated chips on the example's input, columns by the "
                   "restated layouter, advice in pinned host memory, proof bytes out; prove_s excludes the (host, serial) witness "
                   "generation and reading the pk, which are listed under host_s / setup_s")
    return res


def bench_real_flow_multi(h, torch, n_dev, name="kmeans"):
    """one real proof of the kmeans example with h2v_init(devices 0 .. n_dev - 1): create_proof's commit and transform
    batches are cut into one block of columns per device (peer copies over NVLink); the bytes equal the 1-GPU proof's"""
    import numpy as np
    from halo2_vectordb_b200 import circuit as Z
    k, bits = Z.EXAMPLE_PARAMS[name]
    n = 1 << k
    builder = Z.GateThreadBuilder(bits)
    public = []
    Z.EXAMPLES[name](builder.main(0), Z.example_input(name), public)
    builder.make_public(public)
    rc = Z.RangeCircuit(builder, k)
    A = len(rc.advice)
    pinned = torch.empty((A, n, 4), dtype=torch.int64).pin_memory()
    adv = pinned.numpy().view(np.uint64)
    for i, c in enumerate(rc.advice):
        adv[i] = c
    cols = [adv[i] for i in range(A)]
    out = {}
    ref = None
    for devs in ([0], list(range(n_dev))):
        h.init(devs)
        srs = h.ParamsKZG.gen_srs(k)
        pk = h.ProvingKey(srs, rc.cs, rc.fixed, rc.sigma, np.array([k, 0, 0, 0], dtype=np.uint64))
        proof = pk.create_proof(cols, rc.instances, bytes(32))
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            pk.create_proof(cols, rc.instances, bytes(32))
            ts.append(time.perf_counter() - t0)
        if ref is None:
            ref = proof
        out[f"{len(devs)}_gpu"] = {"prove_s": min(ts), "phase_ms": {kk: round(v, 1) for kk, v in pk.last_phase_ms().items()},
                                   "same_bytes_as_1_gpu": proof == ref}
        pk.close()
        srs.close()
    out["example"] = f"{name} k={k}"
    out["speed_up"] = out["1_gpu"]["prove_s"] / out[f"{n_dev}_gpu"]["prove_s"] if n_dev > 1 else 1.0
    rc.close()
    builder.close()
    return out


def _calls(adv, lk, fixed_consts=1):
    """hot-path calls of one proof (SURVEY.md App. C's formulas) from the column counts: commit_lagrange / commit,
    lagrange_to_coeff, coeff_to_extended"""
    a, sets = adv + lk, -(-(adv + lk + fixed_consts + 1) // 2)
    return a + 3 * lk + sets + 6, a + 3 * lk + sets, a + 1 + 3 * lk + sets


PROVE_SHAPES = {   # hot-path call counts per proof from the EXACT column counts of the restated chips + layouter
    # (tests/test_circuit.py; sift_k20: oracle/mock.py's cell count of nearest_vector + merkle_commitment over 1024 x 128
    # vectors at LOOKUP_BITS = 19: 202 518 253 advice cells, 8 921 058 lookup cells); last entry: columns per batch
    "distances_k13": (13, *_calls(9, 2), 32),
    "query_k13": (13, *_calls(147, 19), 160),
    "kmeans_k16": (16, *_calls(535, 72), 96),
    "sift_k20": (20, *_calls(194, 9), 8),
}


def bench_prove_shaped(h, torch, dev, srs16, d_cols16, cols16):
    """The hot-path call schedule of ONE proof of each BASELINE circuit (SURVEY.md App. C: commit_lagrange,
    lagrange_to_coeff and coeff_to_extended per column, one fused divide_by_vanishing + extended_to_coeff) on
    device-resident synthetic uniform columns.  A PROXY for create_proof: witness generation, lookup sorting,
    evaluate_h, evaluations and the transcript are not part of the path and not included."""
    res = {}
    for name, (k, n_msm, n_intt, n_cntt, bcols) in PROVE_SHAPES.items():
        n = 1 << k
        if k == K:
            srs, d_cols, bcols = srs16, d_cols16, cols16
        else:
            srs = h.ParamsKZG(k, None, h.synthetic_bases(n, SYN_A, SYN_B))
            g = torch.Generator(device="cpu").manual_seed(k)
            a = torch.randint(-(1 << 63), (1 << 63) - 1, (bcols, n, 4), dtype=torch.int64, generator=g)
            a[..., 3] &= (1 << 60) - 1
            d_cols = a.to(dev)
        dom = h.EvaluationDomain(4, k)
        d_out = torch.zeros((bcols, 8), dtype=torch.int64, device=dev)
        d_coef = torch.empty_like(d_cols)
        ext_cols = max(1, min(bcols, (1 << 30) // (4 * n * 32)))
        d_ext = torch.empty((ext_cols, 4 * n, 4), dtype=torch.int64, device=dev)
        d_h = torch.empty((1, 4 * n, 4), dtype=torch.int64, device=dev)

        def run():
            left = n_msm
            while left > 0:
                c = min(bcols, left)
                srs.commit_batch_dev(d_cols.data_ptr(), n, c, n, d_out.data_ptr())
                left -= c
            left = n_intt
            while left > 0:
                c = min(bcols, left)
                dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_cols.data_ptr(), n, d_coef.data_ptr(), n, c)
                left -= c
            left = n_cntt
            while left > 0:
                c = min(ext_cols, left)
                dom.transform_dev(h.OP_COEFF_TO_EXTENDED, d_coef.data_ptr(), n, d_ext.data_ptr(), 4 * n, c)
                left -= c
            dom.transform_dev(h.OP_DIVIDE_BY_VANISHING, d_ext.data_ptr(), 4 * n, d_h.data_ptr(), 4 * n, 1)

        run()
        ts = []
        for _ in range(3):
            torch.cuda.synchronize()
            t = time.perf_counter()
            run()
            torch.cuda.synchronize()
            ts.append(time.perf_counter() - t)
        res[name] = {"latency_s": statistics.median(ts), "k": k, "commit_lagrange": n_msm, "lagrange_to_coeff": n_intt,
                     "coeff_to_extended": n_cntt}
        dom.close()
        if k != K:
            srs.close()
            del d_cols
        del d_ext, d_h, d_coef
    res["note"] = "hot-path proxy for one create_proof per circuit (call counts from the exact column counts of the restated chips, App. C's formulas), uniform scalars, device-resident"
    res["latency_s"] = res["kmeans_k16"]["latency_s"]
    res["kmeans_k16_host_facing_s"] = prove_shaped_host(h, torch, srs16)
    res["kmeans_k16_host_in_quotient_on_device_s"] = prove_shaped_resident(h, torch, dev, srs16)
    res["kmeans_k16_all_built_steps"] = prove_shaped_full(h, torch, dev, srs16, d_cols16)
    return res


def prove_shaped_full(h, torch, dev, srs, d_cols):
    """Every create_proof step this library covers, in the order of SURVEY.md 3.1, for the kmeans k = 16 shape
    (App. C estimates: 617 advice + lookup-advice columns, 71 lookups, 310 permutation products): commits, the lookup
    permutations, grand products, lagrange_to_coeff, coeff_to_extended + evaluate_h row loops, the divided quotient and
    its commits, the evaluations at x * omega^rot and the SHPLONK quotient (kate_division + commits).  Columns are
    synthetic and device-resident except where the entry point is host-facing (kate_division: host arrays, PCIe
    included).  Still a PROXY: witness generation, the transcript and the assembly of the product
    numerators / SHPLONK polynomials are not part of it."""
    import numpy as np
    n, ne, bc = N, 4 * N, 96
    n_adv, n_look, n_perm = 617, 71, 310
    dom = h.EvaluationDomain(4, K)
    d_out = torch.zeros((bc, 8), dtype=torch.int64, device=dev)
    d_coef = d_cols.flip(0).contiguous()         # a second set of non-zero columns (denominators), later the coefficient buffer
    d_gp = torch.empty_like(d_cols)
    d_ext = torch.empty((bc, ne, 4), dtype=torch.int64, device=dev)
    d_h = torch.zeros((ne, 4), dtype=torch.int64, device=dev)
    d_hq = torch.empty((ne, 4), dtype=torch.int64, device=dev)
    d_pts = d_cols[0, :2].contiguous()
    d_ev = torch.zeros((bc, 2, 4), dtype=torch.int64, device=dev)
    u = n - 6
    vals = torch.zeros((u, 4), dtype=torch.int64)
    vals[:, 0] = torch.randint(0, 1 << 15, (u,), dtype=torch.int64)
    tab = torch.zeros((u, 4), dtype=torch.int64)
    tab[: 1 << 15, 0] = torch.arange(1 << 15, dtype=torch.int64)
    from halo2_vectordb_b200.synthetic import to_mont      # setup only: Montgomery form of the small lookup values
    m_in = torch.from_numpy(to_mont(vals.numpy().view(np.uint64)).view(np.int64)).to(dev)
    m_tab = torch.from_numpy(to_mont(tab.numpy().view(np.uint64)).view(np.int64)).to(dev)
    d_pa, d_ps = torch.empty_like(m_in), torch.empty_like(m_in)
    hnum = d_cols[1].cpu().pin_memory().numpy().view(np.uint64)
    y = hnum[:3]
    spans = {}

    def span(name, fn):
        torch.cuda.synchronize()
        t = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        spans[name] = spans.get(name, 0.0) + time.perf_counter() - t

    def batches(total):
        return [min(bc, total - i) for i in range(0, total, bc)]

    def commits(total):
        for c in batches(total):
            srs.commit_batch_dev(d_cols.data_ptr(), n, c, n, d_out.data_ptr())

    def run():
        spans.clear()
        span("commit_lagrange advice", lambda: commits(n_adv))
        span("permute_expression_pair", lambda: [h.permute_expression_pair_dev(m_in.data_ptr(), m_tab.data_ptr(), u, d_pa.data_ptr(), d_ps.data_ptr())
                                                 for _ in range(n_look)])
        span("commit_lagrange lookups", lambda: commits(2 * n_look))
        span("grand_product", lambda: [h.grand_product_dev(d_cols.data_ptr(), d_coef.data_ptr(), n, c, d_gp.data_ptr())
                                       for c in batches(n_perm + n_look)])
        span("commit_lagrange products + random + h + shplonk", lambda: commits(n_perm + n_look + 1 + 3 + 2))
        total = n_adv + 2 * n_look + n_perm + n_look

        def transforms():
            for c in batches(total):
                dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_cols.data_ptr(), n, d_coef.data_ptr(), n, c)
                dom.transform_dev(h.OP_COEFF_TO_EXTENDED, d_coef.data_ptr(), n, d_ext.data_ptr(), ne, c)
                dom.quotient_gates(d_h.data_ptr(), y[0], c // 2, d_ext.data_ptr(), ne, d_ext.data_ptr(), ne)
                dom.quotient_permutation(d_h.data_ptr(), y[0], y[1], y[2], c // 2, 2, d_ext.data_ptr(), ne, d_ext.data_ptr(), ne,
                                         d_ext.data_ptr(), ne, d_ext[0].data_ptr(), d_ext[1].data_ptr(), d_ext[2].data_ptr(), 5)
            e = lambda i: d_ext[i].data_ptr()
            for _ in range(n_look):
                dom.quotient_lookup(d_h.data_ptr(), y[0], y[1], y[2], e(3), e(4), e(5), e(6), e(7), e(0), e(1), e(2))
            dom.transform_dev(h.OP_DIVIDE_BY_VANISHING, d_h.data_ptr(), ne, d_hq.data_ptr(), ne, 1)

        span("lagrange_to_coeff + coeff_to_extended + evaluate_h + divide", transforms)
        span("eval_polynomial", lambda: [h._check(h.lib().h2v_eval_polynomial_dev(d_coef.data_ptr(), n, c, n, d_pts.data_ptr(), 2, d_ev.data_ptr()))
                                         for c in batches(total)])
        span("kate_division (host-facing)", lambda: [h.kate_division(hnum, y[0]) for _ in range(4)])
        return sum(spans.values())

    run()
    t = min(run(), run())
    dom.close()
    return {"latency_s": t, "spans_s": {k: round(v, 5) for k, v in spans.items()},
            "note": "kmeans k=16 shape (App. C estimates), every create_proof step the library covers; proxy"}


def prove_shaped_resident(h, torch, dev, srs):
    """The kmeans k=16 schedule with the quotient evaluation on the device as well (SURVEY.md 8(f) row 1): every
    column is uploaded ONCE from pinned host memory (2 MiB), committed, brought to coefficient form, extended and
    folded into h by the gate / permutation kernels without leaving HBM; only the commitments and the divided
    quotient (3n coefficients) come back.  Selector / sigma / z columns reuse the extended buffers (timing only)."""
    import numpy as np
    k, n_msm, n_intt, n_cntt, _ = PROVE_SHAPES["kmeans_k16"]
    bc = int(os.environ.get("H2V_BENCH_BC", "96"))
    g = torch.Generator(device="cpu").manual_seed(6)
    hin = torch.randint(-(1 << 63), (1 << 63) - 1, (bc, N, 4), dtype=torch.int64, generator=g)
    hin[..., 3] &= (1 << 60) - 1
    hin = hin.pin_memory()
    hq = torch.empty((3 * N, 4), dtype=torch.int64).pin_memory()
    dom = h.EvaluationDomain(4, k)
    ne = 4 * N
    d_in2 = torch.empty((2, bc, N, 4), dtype=torch.int64, device=dev)     # double-buffered uploads
    d_coef = torch.empty((bc, N, 4), dtype=torch.int64, device=dev)
    d_ext = torch.empty((bc, ne, 4), dtype=torch.int64, device=dev)
    d_h = torch.zeros((ne, 4), dtype=torch.int64, device=dev)
    d_hq = torch.empty((ne, 4), dtype=torch.int64, device=dev)
    d_out = torch.zeros((bc, 8), dtype=torch.int64, device=dev)
    hout = torch.empty((bc, 8), dtype=torch.int64).pin_memory()
    y = hin[0, :3].numpy().view(np.uint64)
    L = h.lib()
    import threading

    def upload(slot, c):
        h._check(L.h2v_dev_upload(d_in2[slot].data_ptr(), hin.data_ptr(), c * N * 32))

    def run():
        batches = [min(bc, n_msm - i) for i in range(0, n_msm, bc)]
        upload(0, batches[0])
        for i, c in enumerate(batches):
            nxt = None
            if i + 1 < len(batches):        # the next batch crosses PCIe while this one is being processed
                nxt = threading.Thread(target=upload, args=((i + 1) & 1, batches[i + 1]))
                nxt.start()
            d_in = d_in2[i & 1]
            srs.commit_batch_dev(d_in.data_ptr(), N, c, N, d_out.data_ptr())
            h._check(L.h2v_dev_download(hout.data_ptr(), d_out.data_ptr(), c * 64))
            dom.transform_dev(h.OP_LAGRANGE_TO_COEFF, d_in.data_ptr(), N, d_coef.data_ptr(), N, c)
            dom.transform_dev(h.OP_COEFF_TO_EXTENDED, d_coef.data_ptr(), N, d_ext.data_ptr(), ne, c)
            dom.quotient_gates(d_h.data_ptr(), y[0], c, d_ext.data_ptr(), ne, d_ext.data_ptr(), ne)
            dom.quotient_permutation(d_h.data_ptr(), y[0], y[1], y[2], c, 2, d_ext.data_ptr(), ne, d_ext.data_ptr(), ne,
                                     d_ext.data_ptr(), ne, d_ext[0].data_ptr(), d_ext[1].data_ptr(), d_ext[2].data_ptr(), 5)
            if nxt is not None:
                nxt.join()
        dom.transform_dev(h.OP_DIVIDE_BY_VANISHING, d_h.data_ptr(), ne, d_hq.data_ptr(), ne, 1)
        h._check(L.h2v_dev_download(hq.data_ptr(), d_hq.data_ptr(), 3 * N * 32))

    run()
    ts = []
    for _ in range(2):
        torch.cuda.synchronize()
        t = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t)
    dom.close()
    return min(ts)


def prove_shaped_host(h, torch, srs):
    """The kmeans k=16 schedule again, but every column crosses PCIe the way a drop-in under today's create_proof
    would move it (columns live in pinned host memory, evaluate_h stays on the CPU): commit_lagrange batches upload
    the columns, lagrange_to_coeff uploads and downloads them, coeff_to_extended downloads 4x the data."""
    import ctypes as C
    import numpy as np
    k, n_msm, n_intt, n_cntt, _ = PROVE_SHAPES["kmeans_k16"]
    bc = 32
    g = torch.Generator(device="cpu").manual_seed(5)
    hin = torch.randint(-(1 << 63), (1 << 63) - 1, (bc, N, 4), dtype=torch.int64, generator=g)
    hin[..., 3] &= (1 << 60) - 1
    hin = hin.pin_memory()
    hcoef = torch.empty((bc, N, 4), dtype=torch.int64).pin_memory()
    hext = torch.empty((bc, 4 * N, 4), dtype=torch.int64).pin_memory()
    hout = np.zeros((bc, 8), dtype=np.uint64)
    ia = (C.c_void_p * bc)(*[hin[i].data_ptr() for i in range(bc)])
    ca = (C.c_void_p * bc)(*[hcoef[i].data_ptr() for i in range(bc)])
    ea = (C.c_void_p * bc)(*[hext[i].data_ptr() for i in range(bc)])
    dom = h.EvaluationDomain(4, k)
    L = h.lib()

    def run():
        left = n_msm
        while left > 0:
            c = min(bc, left)
            h._check(L.h2v_commit_batch(srs._h, h.H2V_BASIS_LAGRANGE, ia, c, N, hout.ctypes.data_as(C.c_void_p)))
            left -= c
        left = n_intt
        while left > 0:
            c = min(bc, left)
            h._check(L.h2v_domain_transform_batch(dom._h, h.OP_LAGRANGE_TO_COEFF, ia, ca, c))
            left -= c
        left = n_cntt
        while left > 0:
            c = min(bc, left)
            h._check(L.h2v_domain_transform_batch(dom._h, h.OP_COEFF_TO_EXTENDED, ca, ea, c))
            left -= c

    run()
    ts = []
    for _ in range(2):
        t = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t)
    dom.close()
    return min(ts)


def bench_row2(h, torch, dev, d_cols, cols):
    """eval_polynomial (SURVEY.md 8(f) row 2) on the same columns: every column at 3 points, device-resident;
    beside it the oracle's single-threaded Horner on one column (kind "port")."""
    import numpy as np
    from oracle import oracle as O
    pts = d_cols[0, :3].contiguous()
    out = torch.zeros((cols, 3, 4), dtype=torch.int64, device=dev)
    ms = []
    for i in range(6):
        h._check(h.lib().h2v_eval_polynomial_dev(d_cols.data_ptr(), N, cols, N, pts.data_ptr(), 3, out.data_ptr()))
        if i >= 2:
            ms.append(h.last_kernel_ms()["ntt"])       # the polynomial kernels report under class 7
    t = statistics.median(ms) * 1e-3
    col0 = d_cols[0].cpu().numpy().view(np.uint64)
    x0 = pts[0].cpu().numpy().view(np.uint64)
    assert (O.fr_eval_poly(col0, x0) == out[0, 0].cpu().numpy().view(np.uint64)).all()
    t0 = time.perf_counter()
    for _ in range(4):
        O.fr_eval_poly(col0, x0)
    cpu = 4 * N / (time.perf_counter() - t0)
    # permute_expression_pair (lookup argument, create_proof step 5): 2^16 - 6 usable rows of a LOOKUP_BITS = 15 range lookup
    u, bits = N - 6, 15
    g = torch.Generator(device=dev).manual_seed(17)
    vals = torch.zeros((u, 4), dtype=torch.int64, device=dev)
    vals[:, 0] = torch.randint(0, 1 << bits, (u,), dtype=torch.int64, generator=g, device=dev)
    tab = torch.zeros((u, 4), dtype=torch.int64, device=dev)
    tab[: 1 << bits, 0] = torch.arange(1 << bits, dtype=torch.int64, device=dev)
    # inputs must be Montgomery: convert the small canonical values on the device once (setup, untimed)
    from halo2_vectordb_b200.synthetic import to_mont
    m_in = torch.from_numpy(to_mont(vals.cpu().numpy().view(np.uint64)).view(np.int64)).to(dev)
    m_tab = torch.from_numpy(to_mont(tab.cpu().numpy().view(np.uint64)).view(np.int64)).to(dev)
    o_a, o_s = torch.empty_like(m_in), torch.empty_like(m_in)
    pm = []
    for i in range(6):
        h.permute_expression_pair_dev(m_in.data_ptr(), m_tab.data_ptr(), u, o_a.data_ptr(), o_s.data_ptr())
        if i >= 2:
            pm.append(h.last_kernel_ms()["ntt"])
    t_p = statistics.median(pm) * 1e-3
    hi, ht = m_in.cpu().numpy().view(np.uint64), m_tab.cpu().numpy().view(np.uint64)
    t0 = time.perf_counter()
    ea, es = O.permute_expression_pair(hi, ht)
    cpu_p = time.perf_counter() - t0
    assert (ea == o_a.cpu().numpy().view(np.uint64)).all() and (es == o_s.cpu().numpy().view(np.uint64)).all()
    return {"eval_polynomial_gcoeff_per_s": cols * 3 * N / t / 1e9, "ms": t * 1e3, "polys": cols, "points": 3,
            "cpu_port_gcoeff_per_s": cpu / 1e9, "cpu_cores": 1,
            "permute_expression_pair": {"rows": u, "ms": t_p * 1e3, "mrows_per_s": u / t_p / 1e6, "cpu_port_ms": cpu_p * 1e3,
                                        "note": "LOOKUP_BITS = 15 range lookup, device-resident; CPU port = oracle qsort, one core"}}


def bench_row1(h, torch, dev):
    """evaluate_h's row loops (SURVEY.md 8(f) row 1) at k = 16, extended_k = 18, device-resident: 128 vertical gates,
    a permutation argument over 128 columns (chunk_len 2) and one lookup, on uniform synthetic extended columns;
    beside them the oracle's scalar loops on a k = 10 domain (kind "port", one core)."""
    import numpy as np
    from oracle import oracle as O
    k, gates = K, 128
    dom = h.EvaluationDomain(4, k)
    ne = 1 << dom.extended_k
    g = torch.Generator(device=dev).manual_seed(11)

    def cols_dev(c):
        a = torch.randint(-(1 << 63), (1 << 63) - 1, (c, ne, 4), dtype=torch.int64, generator=g, device=dev)
        a[..., 3] &= (1 << 60) - 1
        return a

    d_q, d_a, d_sig, d_z, d_misc = cols_dev(gates), cols_dev(gates), cols_dev(gates), cols_dev(gates // 2), cols_dev(9)
    d_h = torch.zeros((ne, 4), dtype=torch.int64, device=dev)
    y = d_misc[0, :3].cpu().numpy().view(np.uint64)
    m = lambda i: d_misc[i].data_ptr()

    def timed(fn):
        ms = []
        for i in range(6):
            fn()
            if i >= 2:
                ms.append(h.last_kernel_ms()["ntt"])       # the quotient kernels report under class 7
        return statistics.median(ms) * 1e-3

    t_g = timed(lambda: dom.quotient_gates(d_h.data_ptr(), y[0], gates, d_q.data_ptr(), ne, d_a.data_ptr(), ne))
    t_p = timed(lambda: dom.quotient_permutation(d_h.data_ptr(), y[0], y[1], y[2], gates, 2, d_a.data_ptr(), ne, d_sig.data_ptr(), ne,
                                                 d_z.data_ptr(), ne, m(1), m(2), m(3), 5))
    t_l = timed(lambda: dom.quotient_lookup(d_h.data_ptr(), y[0], y[1], y[2], m(4), m(5), m(6), m(7), m(8), m(1), m(2), m(3)))
    dom.close()
    # CPU port on a small domain, one core
    ck, cg = 10, 8
    od = O.EvaluationDomain(4, ck)
    cne = 1 << od.extended_k
    ca = O.fr_fill(cg * cne, 3).reshape(cg, cne, 4)
    cz = O.fr_fill((cg // 2) * cne, 4).reshape(cg // 2, cne, 4)
    ch = np.zeros((cne, 4), dtype=np.uint64)
    t0 = time.perf_counter()
    od.quotient_gates(ch, y[0], ca, ca)
    c_g = cg * cne / (time.perf_counter() - t0)
    t0 = time.perf_counter()
    od.quotient_permutation(ch, y[0], y[1], y[2], 2, ca, ca, cz, ca[0], ca[1], ca[2], 5)
    c_p = cg * cne / (time.perf_counter() - t0)
    # products per row: 3 per gate, 4 per permuted column + 2.5 per grand product, 13 per lookup
    n_adv = PROVE_SHAPES["kmeans_k16"][4]
    return {"gate_rows_per_s": gates * ne / t_g, "perm_col_rows_per_s": gates * ne / t_p, "lookup_rows_per_s": ne / t_l,
            "ms": {"gates_128": t_g * 1e3, "permutation_128": t_p * 1e3, "lookup_1": t_l * 1e3},
            "fr_mul_per_s": {"gates": 3 * gates * ne / t_g, "permutation": (4 * gates + 2.5 * gates / 2 + 4) * ne / t_p},
            "dram_gb_per_s": {"gates": (2 * gates + 2) * ne * 32 / t_g / 1e9, "permutation": (2.5 * gates + 5) * ne * 32 / t_p / 1e9},
            "cpu_port": {"gate_rows_per_s": c_g, "perm_col_rows_per_s": c_p, "cores": 1, "sample": f"k={ck}, {cg} columns, oracle scalar loops"},
            "note": f"k={k}, extended_k={dom.extended_k}, uniform synthetic extended columns resident in HBM; per-term rates, {n_adv} advice columns in the kmeans batch"}


def bench_witness(h, torch, dev, srs, peak):
    """Same commit batch on witness-shaped scalars (60% {0,1}, 30% < 2^15, 10% full width / r - small): the
    distribution FixedPointChip columns really have (/root/reference/src/gadget/fixed_point.rs:68-119).  The second
    headline: per-kernel-class times, the share of the step outside msm_accumulate, and the accumulate kernel's roofline
    on the mixed additions it actually executes (one per non-zero digit: sorted entries, read back from the histogram)."""
    import numpy as np
    from halo2_vectordb_b200.synthetic import witness_like
    cols = 96
    a = torch.from_numpy(witness_like(cols, N, 15, 7).view(np.int64)).to(dev)
    out = torch.zeros((cols, 8), dtype=torch.int64, device=dev)
    ms, kms = [], {}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(8):
        e0.record()
        srs.commit_batch_dev(a.data_ptr(), N, cols, N, out.data_ptr())      # blocks until the result is there
        e1.record()
        e1.synchronize()
        if i >= 2:
            k = h.last_kernel_ms()
            ms.append(e0.elapsed_time(e1))
            for kk, v in k.items():
                kms.setdefault(kk, []).append(v)
    t = statistics.median(ms) * 1e-3
    kmed = {kk: statistics.median(v) for kk, v in kms.items()}
    c, w = srs.info()
    # non-zero digits of the batch under the window the call used, counted on the host from the same scalars
    acc_s = kmed["msm_accumulate"] * 1e-3
    res = {"msm_mpts_per_s": cols * N / t / 1e6, "ms_per_step": t * 1e3, "cols_per_step": cols, "lookup_bits": 15,
           "kernel_ms_per_step": {kk: round(v, 4) for kk, v in kmed.items() if v},
           # the step time is the wall clock of the call (CUDA events around it); the share is the part of it not covered
           # by the accumulate kernel
           "non_accumulate_share": max(0.0, 1.0 - kmed["msm_accumulate"] * 1e-3 / t),
           "kernel_span_sum_ms": sum(kmed.values()),
           "window_bits": c, "windows": w}
    entries = h.last_msm_entries()
    if entries and acc_s > 0:
        res["roofline"] = {"bound": "int32-pipe (IMAD.WIDE)", "kernel": "msm_accumulate_kernel", "unit": "T wide-MAC/s",
                           "executed": entries * MIXED_ADD_MACS / acc_s / 1e12, "peak": peak / 1e12, "frac": entries * MIXED_ADD_MACS / acc_s / peak,
                           "mixed_additions_per_launch": int(entries)}
    return res


def bench_ntt(h, torch, dev, peak):
    """Fr NTT throughput on the same circuit shape: lagrange_to_coeff (2^16) and coeff_to_extended (2^16 -> 2^18)."""
    import json as _json
    try:
        hbm = _json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        hbm_src = "MEASURED_PEAKS.json"
    except Exception:
        hbm, hbm_src = 6650.0, "fallback"
    dom = h.EvaluationDomain(4, K)
    cols = 64
    g = torch.Generator(device="cpu").manual_seed(99)
    a = torch.randint(-(1 << 63), (1 << 63) - 1, (cols, N, 4), dtype=torch.int64, generator=g)
    a[..., 3] &= (1 << 60) - 1
    d_in = a.to(dev)
    d_n = torch.empty_like(d_in)
    d_ext = torch.empty((cols, 4 * N, 4), dtype=torch.int64, device=dev)
    res = {}
    for name, op, src, dst, ostride, L in (("lagrange_to_coeff", h.OP_LAGRANGE_TO_COEFF, d_in, d_n, N, K),
                                           ("coeff_to_extended", h.OP_COEFF_TO_EXTENDED, d_in, d_ext, 4 * N, K + 2)):
        for _ in range(3):
            dom.transform_dev(op, src.data_ptr(), N, dst.data_ptr(), ostride, cols)
        ms = []
        for _ in range(10):
            dom.transform_dev(op, src.data_ptr(), N, dst.data_ptr(), ostride, cols)
            ms.append(h.last_kernel_ms()["ntt"])
        t = statistics.median(ms) * 1e-3
        size = 1 << L
        passes = (L + 8) // 9
        alg_bytes = 64 * size * passes * cols
        # SURVEY.md 8(d): work(n) = (n/2) log2 n x 136 wide-MACs, + n x 136 for the iNTT / coset scaling (n = the elements
        # that are scaled: every output of lagrange_to_coeff, the N input coefficients of coeff_to_extended)
        bfly_macs = (size // 2) * L * FQ_MUL_MACS * cols
        alg_macs = bfly_macs + N * FQ_MUL_MACS * cols
        # what the kernel executes: stage 0 has unit twiddles, 3 of the 8 products of the first radix-8 round are by 1, the
        # 1/n of lagrange_to_coeff is one word of Montgomery reduction (8 wide-MACs) instead of a product; zero-padded
        # input (coeff_to_extended) turns the first two stages into broadcasts and leaves 3 products in the first round
        # A twiddle product is Shoup's (csrc/shoup.cuh): 99 IMAD.WIDE + 16 low-only IMAD (half the pipe time) = 107
        # wide-MAC equivalents instead of the 136 of a Montgomery product.
        if name == "lagrange_to_coeff":
            exec_macs = ((size // 2) * (L - 1) - 3 * (size // 8)) * SHOUP_MUL_MACS * cols + 8 * size * cols
        else:
            exec_macs = ((size // 2) * (L - 2) - (size // 8)) * SHOUP_MUL_MACS * cols + N * FQ_MUL_MACS * cols
        res[name] = {"gelem_per_s": cols * size / t / 1e9, "ms": t * 1e3, "cols": cols, "log_n": L,
                     "roofline": {"bound": "hbm", "achieved": alg_bytes / t / 1e9, "peak": hbm, "unit": "GB/s",
                                  "frac": alg_bytes / t / 1e9 / hbm, "peak_source": hbm_src,
                                  # both passes of lagrange_to_coeff 2^16 x 64: 134.3 + 89.6 and 136.4 + 88.8 MB read + written
                                  # (ncu --set full, profiles/r02_final2_ncu_summary.txt) against 537 MB algorithmic
                                  "traffic": 4.49e8 if name == "lagrange_to_coeff" else None},
                     "roofline_int": {"achieved": alg_macs / t / 1e12, "peak": peak / 1e12, "unit": "T wide-MAC/s",
                                      "frac": alg_macs / t / peak, "frac_butterflies_only": bfly_macs / t / peak,
                                      "frac_executed": exec_macs / t / peak,
                                      "algorithmic": "SURVEY.md 8(d): ((n/2) log2 n + scaled elements) x 136 wide-MACs",
                                      "executed": "twiddle products by Shoup's method: 107 wide-MAC equivalents each (99 IMAD.WIDE + 16 IMAD), unit twiddles skipped"}}
    # end to end through the host-facing batch entry point: pinned host columns in, pinned host columns out
    import ctypes as C
    import numpy as np
    hin = a[:32].contiguous().pin_memory()
    hout = torch.empty((32, 4 * N, 4), dtype=torch.int64).pin_memory()
    ia = (C.c_void_p * 32)(*[hin[i].data_ptr() for i in range(32)])
    for name, op, rows in (("lagrange_to_coeff", h.OP_LAGRANGE_TO_COEFF, N), ("coeff_to_extended", h.OP_COEFF_TO_EXTENDED, 4 * N)):
        oa = (C.c_void_p * 32)(*[hout[i].data_ptr() for i in range(32)])
        ts = []
        for i in range(8):
            t0 = time.perf_counter()
            h._check(h.lib().h2v_domain_transform_batch(dom._h, op, ia, oa, 32))
            ts.append(time.perf_counter() - t0)
        t = statistics.median(ts[3:])
        res[name]["e2e"] = {"gelem_per_s": 32 * rows / t / 1e9, "ms": t * 1e3, "cols": 32,
                            "h2d_bytes": 32 * N * 32, "d2h_bytes": 32 * rows * 32}
    dom.close()
    return res


if __name__ == "__main__":
    main()
