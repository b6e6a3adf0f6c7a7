#!/usr/bin/env python3
"""bench.py — Groth16 constraints/sec on synthetic R1CS, N GPUs of one node.

    python bench.py --gpus N --steps K --warmup W            # this repo (libzkb200.so, sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm on the host cores, SAME circuit
    python bench.py --curve bls12_381 --log-n 22 --gpus 8    # BASELINE.json config 4
    python bench.py --steps K --dump-outputs DIR             # also write the proof of the last timed step under DIR

Workload (default = BASELINE.json config 3): synthetic R1CS with 2^20 - 2 constraints, one public input, so the
evaluation domain is exactly 2^20; uniform 252-bit witness (MSM worst case), BN254.  A "step" is one proof:
witness_map (3 SpMV + 7 NTT) + 4 G1 MSM + 1 G2 MSM + final combination.
  value : whole-job constraints/s with z, the CSR matrices and the proving key resident in HBM
  e2e   : the same through the C-ABI call a `zokrates_b200` Rust shim makes (zkb_groth16_prove): z in pinned
          host memory, H2D of z and D2H of the window sums / proof inside the timed region
Multi-GPU: every MSM is sharded by index range over the ranks (no data-path collective); the 5 partial
sums per rank are all-gathered (NCCL) and rank 0 finishes the proof; the witness map is replicated for N <= 2 and
its three chains are computed once each and broadcast (NCCL over NVLink) for N >= 3.
The reference arm times oracle/libzkoracle.so — the C restatement of ark's prover (the reference is
Rust + un-vendored arkworks crates and cannot be built here, see DESIGN.md) — on all host threads (team size set
explicitly from the usable core count: torchrun exports OMP_NUM_THREADS=1), on the SAME circuit, key, witness, steps and
warm-up as the GPU arm; circuit and key are generated on the CPU (no kernel of this repo runs in that arm).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = 20
TRAPDOOR = [0x1111, 0x2222, 0x3333, 0x4444, 0x123456789ABCDEF, 3, 7]
R_S = (1234567, 7654321)
CPU_SAMPLE_MAX_LOG_N = 20  # cpu_baseline leg of the GPU arm: the bench circuit itself up to 2^20, a 2^20 circuit of the same family above
CURVE_IDS = {"bn128": 0, "bls12_381": 1}
MADS_PER_MUL = {"bn128": 136, "bls12_381": 300}   # 2 L^2 + L wide multiply-adds per Montgomery multiplication (SURVEY.md §8d)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md).  Started before the warm-up (nvidia-smi takes a few
    hundred ms to come up, longer than a short timed region); every sample carries the host time it was read at and
    only those inside the marked timed windows are reported (all load samples if a window caught none)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0, period_ms=50):
        self.index, self.period_ms, self.proc, self.lines, self.windows = index, period_ms, None, [], []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", str(self.period_ms), "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line))

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if self.proc:
            time.sleep(2.5 * self.period_ms / 1e3)
            self.proc.terminate()
        rows = []
        for ts, line in self.lines:
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                rows.append((ts, float(p[1]), float(p[2]), float(p[3]), p[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if any(a <= r[0] <= b + self.period_ms / 1e3 for a, b in self.windows)]
        scope = "timed region"
        if not inside:                       # fall back to the samples taken under load (warm-up + timed steps)
            inside = [r for r in rows if r[3] > 250.0] or rows
            scope = "warm-up + timed steps (no sample fell inside the timed windows)"
        reasons = set()
        for r in inside:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm = [r[1] for r in inside]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max((r[2] for r in inside), default=None),
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope,
                "power_w_max": max((r[3] for r in inside), default=None)}


def load_oracle():
    """CPU checker / baseline (oracle/libzkoracle.so).  Only the cpu_baseline leg and --impl reference use it."""
    import __graft_entry__ as g
    from tests.oracle_c import OracleC
    oc = OracleC(g.build_oracle())
    # team size = min(online CPUs, affinity mask, cgroup CPU quota) decided inside the library (zko_pool_threads) and NOT from
    # OMP_NUM_THREADS: torchrun exports OMP_NUM_THREADS=1 to every rank, which starved this arm in round 1
    os.environ.pop("OMP_NUM_THREADS", None)
    return oc


class CpuFieldOps:
    """`field_op` of the synthetic generator served by the CPU oracle (the reference arm runs no kernel of this repo)."""

    def __init__(self, oc, cid):
        self.oc, self.cid = oc, cid

    def field_op(self, field, op, a, b):
        return self.oc.field_op(self.cid, field, op, a, b)


def dump_outputs(out_dir, proof, fq_bytes):
    """The proof a caller receives (A in G1, B in G2, C in G1) as DIR/proof_{a,b,c}.npy.  A coordinate is a 256- or
    384-bit field element, so it is stored as 16-bit little-endian limbs in float64, which hold it exactly."""
    os.makedirs(out_dir, exist_ok=True)
    limbs = np.frombuffer(proof, dtype="<u2").astype(np.float64).reshape(8, fq_bytes // 2)
    for name, arr in (("proof_a", limbs[0:2]), ("proof_b", limbs[2:6].reshape(2, 2, -1)), ("proof_c", limbs[6:8])):
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def workload_name(args):
    return f"synthetic-r1cs-2^{args.log_n}-{args.curve}-groth16"


def share_wm_for(world):
    # three or more ranks: the witness map's three chains are computed once each and exchanged over NVLink
    return world >= 3 and os.environ.get("ZKB_WM_SHARE", "1") != "0"


def bench_config(args, world, variables):
    """`config` of the JSON line — identical in both arms (the reference arm reports on this arm's config)."""
    n_cons = (1 << args.log_n) - 2
    return {"workload": workload_name(args), "constraints": n_cons, "domain": 1 << args.log_n, "variables": int(variables),
            "witness": args.witness, "curve": args.curve,
            "parallelism": f"msm-index-shard x{world} (work-balanced cuts), witness_map " + ("chains shared over NVLink" if share_wm_for(world) else "replicated"),
            "l2": "inputs larger than L2: the resident proving key (0.4 GB at 2^20 BN254, window tables on top) and the sort buffers are "
                  "streamed every proof, no flush needed",
            "timed_region": "z resident in HBM -> proof bytes on host (e2e: z in pinned host memory -> proof bytes on host)"}


def run_reference(args):
    """The reference's CPU prover (ark-equivalent C port) on the same circuit / key / witness / steps / warm-up."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from zokrates_b200 import synthetic
    cid = CURVE_IDS[args.curve]
    oc = load_oracle()
    fq_bytes = 32 if cid == 0 else 48
    n_cons = (1 << args.log_n) - 2
    t0 = time.perf_counter()
    r1cs, z = synthetic.make_layered(CpuFieldOps(oc, cid), args.curve, n_cons, distribution=args.witness)
    pk = oc.setup(cid, r1cs, TRAPDOOR)
    prep_s = time.perf_counter() - t0
    times, stage = [], None
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        proof, stage = oc.prove(cid, pk, r1cs, z, *R_S, fq_bytes)
        dt = time.perf_counter() - t
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, proof, fq_bytes)
    total = sum(times)
    value = n_cons * len(times) / total
    line = {
        "impl": "reference", "metric": "groth16_constraints_per_sec", "value": value, "unit": "constraints/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u256-montgomery" if cid == 0 else "u384-montgomery",
        "data": "synthetic",
        "config": bench_config(args, args.gpus, r1cs.num_variables),
        "reference_timed_region": "proving.key bytes + R1CS + z in host memory -> proof bytes (key deserialisation included, as in "
                                  "zokrates_ark/src/groth16.rs:40-44); no GPU is used whatever --gpus says",
        "cpu_baseline": {"value": value, "unit": "constraints/s", "cores": oc.threads(), "kind": "port",
                         "sample": f"{len(times)} proofs of the full 2^{args.log_n}-2 constraint circuit (ark-equivalent C port of the reference's prover, "
                                   "MSM parallel over windows only as in ark 0.3.0)"},
        "e2e": {"value": value, "unit": "constraints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "stage_s": {k: float(v) for k, v in zip(("pk_deserialize", "witness_map", "msm_g1", "msm_g2", "total"), stage)},
        "prep_s": round(prep_s, 1),
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=LOG_N)
    ap.add_argument("--curve", default="bn128", choices=["bn128", "bls12_381"])
    ap.add_argument("--witness", default="uniform", choices=["uniform", "bits"])
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--table-c", type=int, default=0, help="force the window width of the HBM window tables (0: cost model)")
    ap.add_argument("--opt", action="append", default=[], metavar="ID=VALUE", help="zkb_ctx_set_option(ID, VALUE) before the key is loaded (tuning runs)")
    ap.add_argument("--pipeline", type=int, default=2, choices=[1, 2], help="proofs in flight per GPU (2: submit i+1 before collecting i)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step as DIR/proof_{a,b,c}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)          # timing rule: at least three warm-up steps, in both arms
    if args.impl == "reference":
        return run_reference(args)
    # stdout carries exactly ONE line (the JSON): libraries that print on fd 1 (NCCL's version banner, whatever
    # NCCL_DEBUG / nccl.conf say) go to stderr for the duration of the run
    sys.stdout.flush()
    stdout_fd = os.dup(1)
    os.dup2(2, 1)

    import torch
    import torch.distributed as dist
    from zokrates_b200 import synthetic
    from zokrates_b200._lib import Context, Library

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (libzkb200 has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the launcher set it: fd 1 already points at stderr, so NCCL's banner / INFO lines (which the
        # driver reads to count the ranks) cannot mix with the one JSON line
        # the chain broadcasts run while the accumulate kernels keep every SM full: give NCCL's kernels a high-priority stream
        # (their CTAs are taken first when an SM drains) and few, small CTAs — the exchange is 3 x 32 MB per proof, latency matters
        pg_opts = None
        try:
            pg_opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            if os.environ.get("ZKB_NCCL_MAX_CTAS"):
                pg_opts.config.max_ctas = int(os.environ["ZKB_NCCL_MAX_CTAS"])
        except Exception:                                     # older torch: default options
            pg_opts = None
        kw = {"pg_options": pg_opts} if pg_opts is not None else {}
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local), **kw)

    lib = Library()
    cid = CURVE_IDS[args.curve]
    ctx = Context(cid, local, lib)
    n_cons = (1 << args.log_n) - 2

    # -- untimed preparation: circuit, witness (batched field ops on the GPU), setup, resident key shard
    t_prep = time.perf_counter()
    r1cs, z = synthetic.make_layered(ctx, args.curve, n_cons, distribution=args.witness)
    r1cs_h = ctx.r1cs_load(r1cs.num_constraints, r1cs.num_instance, r1cs.num_witness, r1cs.matrices())
    pk = ctx.setup(r1cs_h, TRAPDOOR)
    setup_ms = ctx.timings()
    if args.table_c:
        from zokrates_b200._lib import OPT_TABLE_C
        ctx.set_option(OPT_TABLE_C, args.table_c)
    for kv in args.opt:
        oid, val = kv.split("=")
        ctx.set_option(int(oid), int(val))
    pk_h = ctx.pk_load(pk, rank, world)
    pk_bytes = len(pk)
    table_info = ctx.pk_table_info(pk_h)
    keep_pk = rank == 0 and args.log_n <= CPU_SAMPLE_MAX_LOG_N and (world == 1 or not args.skip_cpu_baseline)
    if not keep_pk:
        del pk
    z_pinned = torch.from_numpy(z).pin_memory()
    z_host = z_pinned.numpy()
    ctx.set_assignment(r1cs_h, z_host)
    prep_s = time.perf_counter() - t_prep
    r_s = R_S

    dev = torch.device("cuda", local)
    last_stage = {}

    # three or more ranks: the witness map's three chains are computed once each and broadcast over NVLink
    # (zkb_groth16_prove_begin_async / _end_async, zokrates_b200/distributed.py); ZKB_WM_SHARE=0 keeps it replicated
    share_wm = share_wm_for(world)

    # Pipelined proving (include/zkb.h: zkb_groth16_prove_submit / _collect): the whole device work of proof i + 1 is enqueued
    # BEFORE the host collects proof i, so the GPU never idles while the host finishes a proof (last additions of each MSM,
    # final combination, the all_gather of the partial sums).  Every one of the K proofs is submitted and collected inside
    # the timed region.  --pipeline 1 proves strictly one at a time (the latency figure).
    def submit(z_arg):
        if world == 1:
            return ctx.prove_submit(pk_h, r1cs_h, z_arg, *r_s)
        if share_wm:
            from zokrates_b200.distributed import submit_shared_wm
            return submit_shared_wm(ctx, pk_h, r1cs_h, z_arg, device=dev)
        return ctx.prove_submit(pk_h, r1cs_h, z_arg)

    def collect(ticket):
        if world == 1:
            out = ctx.prove_collect(ticket)
            last_stage.update(ctx.timings())
            return out
        from zokrates_b200.distributed import gather_partials
        if rank == 0:
            ctx.finalize_prepare(pk_h, *r_s)           # r*delta1 ... s*delta2 on host threads underneath the gather
        partial = ctx.prove_collect_partial(ticket)
        last_stage.update(ctx.timings())
        allp = gather_partials(partial, device=dev)    # 5 partial sums per rank -> all ranks (NCCL all_gather, < 1 kB each)
        return ctx.finalize(pk_h, allp, world, *r_s) if rank == 0 else None

    def run_steps(z_arg, steps, on_proof):
        depth = max(1, min(args.pipeline, 2))
        pending = []
        proof = None
        for _ in range(steps):
            pending.append(submit(z_arg))
            if len(pending) >= depth:
                proof = collect(pending.pop(0))
                on_proof()
        while pending:
            proof = collect(pending.pop(0))
            on_proof()
        return proof

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(z_arg, steps):
        """K proofs bracketed by barrier + synchronize; CUDA events on the current stream bracket the same region (every proof
        is collected — its device work complete — before the closing event), wall clock and device clock agree; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = ctx.launch_count()
        stage = {}

        def on_proof():
            for k, v in last_stage.items():
                stage[k] = stage.get(k, 0.0) + v
        t0 = time.perf_counter()
        e0.record()
        proof = run_steps(z_arg, steps, on_proof)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        dev_s = e0.elapsed_time(e1) / 1e3
        elapsed = max(wall, dev_s)
        if world > 1:
            tt = torch.tensor([elapsed], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            elapsed = float(tt.item())
        return elapsed, {k: v / steps for k, v in stage.items()}, ctx.launch_count() - launches0, proof

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    run_steps(None, args.warmup, lambda: None)
    tw0 = time.perf_counter()
    t_res, stage_res, launches, proof = timed(None, args.steps)
    sampler.mark(tw0, time.perf_counter())
    run_steps(z_host, 2, lambda: None)
    tw0 = time.perf_counter()
    t_e2e, stage_e2e, _, proof2 = timed(z_host, args.steps)
    sampler.mark(tw0, time.perf_counter())
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and proof != proof2:
        raise SystemExit("resident and e2e proofs differ")
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, proof, ctx.fq_bytes)
    # latency of ONE proof with nothing else in flight (what --pipeline 1 would time), after the throughput runs
    lat = []
    saved_depth = args.pipeline
    args.pipeline = 1
    for _ in range(5):
        barrier()
        t0 = time.perf_counter()
        run_steps(z_host, 1, lambda: None)
        lat.append(time.perf_counter() - t0)
    args.pipeline = saved_depth
    latency_ms = 1e3 * sorted(lat)[len(lat) // 2]

    # the trait-shaped call: `Backend::generate_proof` is static and receives the key BYTES every time
    # (zokrates_ark/src/groth16.rs:40-44), so one call = load the key by content (fingerprint of the bytes, the resident key and
    # its window tables are found again: ZKB_OPT_PK_CACHE) + prove with z in host memory + release the handle.  One proof at a
    # time, nothing in flight.  The R1CS stays loaded (a program cache of the same kind exists behind zkb_prog_load).
    trait_call = None
    if world == 1 and keep_pk:
        tc = []
        for _ in range(5):
            barrier()
            t0 = time.perf_counter()
            h2 = ctx.pk_load(pk, 0, 1)
            hit = "pk_cache_hit" in ctx.timings()
            t1 = time.perf_counter()
            ctx.prove(h2, r1cs_h, z_host, *r_s)
            ctx.pk_free(h2)
            tc.append((time.perf_counter() - t0, t1 - t0, hit))
        tc.sort()
        trait_call = {"ms_per_proof": 1e3 * tc[len(tc) // 2][0], "pk_load_by_content_ms": 1e3 * tc[len(tc) // 2][1], "cache_hit": bool(tc[len(tc) // 2][2]),
                      "key_bytes": pk_bytes,
                      "note": "zkb_pk_load(key bytes) -> fingerprint, cache hit + zkb_groth16_prove(z in host memory) + zkb_pk_free, sequential"}

    value = n_cons * args.steps / t_res
    e2e_value = n_cons * args.steps / t_e2e

    # -- roofline of the dominant kernel: the bucket accumulation of the h_query MSM (no infinity points, uniform scalars,
    #    so the canonical n*W*10 count is not flattered by the infinity-skipping views used for a/b1/b2).  The kernel is
    #    integer-multiply bound (230 MAD per algorithmic byte, far right of the HBM ridge), so the binding resource is the
    #    32x32+64 multiply-add pipe: peak = measured IMAD.WIDE.U32 rate / (2 L^2 + L) MADs per Montgomery multiplication.
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    n_pairs = (r1cs.domain_size - 1) // world            # (scalar, point) pairs one accum1 launch of msm_h processes
    acc_ms = stage_res.get("accum1_g1_h", 0.0)
    roofline = None
    if rank == 0 and acc_ms > 0:
        mads = MADS_PER_MUL[args.curve]
        imad_peak = ctx.peak_probe(0, 40000)             # 32x32+64 multiply-adds per second, dependent-free IMAD.WIDE.U32 chains
        mul_probe = ctx.peak_probe(1, 4000)              # this repo's own register-resident Montgomery multiplication (secondary)
        carry_peak = ctx.peak_probe(2, 10000)            # the same wide MADs carry-chained (IMAD.WIDE.U32.X), as a multiplier issues them
        g1_bytes = 64 if cid == 0 else 96
        alg_bytes = n_pairs * (32.0 + g1_bytes)          # 32 B scalar + one affine point per pair (SURVEY §8d)
        alg_muls = n_pairs * 16 * 10.0                   # canonical: W = 16 windows x 10 Fq-mul per mixed add (SURVEY §8d)
        traffic = None                                   # DRAM bytes per launch from the committed ncu --set full capture
        if cid == 0 and args.log_n == 20:
            try:
                tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))["k_msm_accum1<Fq> (h_query MSM)"]
                traffic = tr["dram_bytes"] / world
            except (OSError, KeyError, ValueError):
                pass
        achieved = alg_muls / (acc_ms * 1e-3)
        peak_mul = imad_peak / mads
        roofline = {"kernel": "k_msm_accum1<Fq> (h_query MSM)", "bound": "int32-mad", "achieved": achieved, "peak": peak_mul,
                    "unit": "Fq-mul/s", "frac": achieved / peak_mul, "traffic": traffic,
                    "peak_source": f"measured in this run: dependent-free IMAD.WIDE.U32 chains (zkb_peak_probe kind 0, {imad_peak:.4g} MAD/s) / {mads} MADs per "
                                   "Montgomery multiplication (SURVEY.md §8d)",
                    "avg_launch_ms": acc_ms, "algorithmic_fq_mul_per_launch": alg_muls, "algorithmic_bytes_per_launch": alg_bytes,
                    "executed_windows": table_info["W_h"] or None,
                    "traffic_note": "ncu dram__bytes_read+write of this kernel: the gathers go to HBM-resident window tables 2^(cw)P, a deliberate "
                                    "bytes-for-multiplications trade (fewer mixed additions per scalar, one bucket set); not binding (about 10 % of HBM peak)",
                    "hbm": {"achieved": alg_bytes / (acc_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": alg_bytes / (acc_ms * 1e-3) / 1e9 / hbm_peak, "peak_source": hbm_src},
                    "carry_chain": {"peak": carry_peak / mads, "unit": "Fq-mul/s", "frac": achieved / (carry_peak / mads), "mad_per_s": carry_peak,
                                    "note": "zkb_peak_probe kind 2: rows of carry-chained wide MADs (1 IMAD.WIDE.U32 + 7 IMAD.WIDE.U32.X); the .X form "
                                            "occupies the fmaheavy pipe longer than the carry-free form of kind 0, and ncu names that pipe as the "
                                            "binding unit of the kernel (sm__pipe_fmaheavy_cycles_active 87.6 %, profiles/r02_ncu_accum1_g2.md)"},
                    "mul_probe": {"peak": mul_probe, "unit": "Fq-mul/s", "frac": achieved / mul_probe,
                                  "note": "this repo's own Fp::mul in a register-resident loop — self-referential, secondary"}}

    # the collectives are over: the other ranks leave, rank 0 has the host cores to itself for the CPU baseline
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return

    # -- CPU baseline: ONE proof of the reference's CPU algorithm on the box's host cores, same circuit / key / witness / r / s
    #    (above 2^20: a 2^20 circuit of the same family), and the checker doing its job: the bytes must equal the GPU's
    cpu_baseline = None
    if rank == 0 and not args.skip_cpu_baseline:
        oc = load_oracle()
        fq_bytes = 32 if cid == 0 else 48
        if args.log_n <= CPU_SAMPLE_MAX_LOG_N:
            c_r1cs, c_z, c_pk, c_n, gpu_proof = r1cs, z, pk, n_cons, proof
            sample = f"1 proof of the bench circuit itself (2^{args.log_n}-2 constraints)"
        else:
            c_n = (1 << CPU_SAMPLE_MAX_LOG_N) - 2
            ctx2 = Context(cid, local, lib)          # full (unsharded) key of the sample circuit on this rank's GPU
            c_r1cs, c_z = synthetic.make_layered(ctx2, args.curve, c_n, distribution=args.witness)
            h2 = ctx2.r1cs_load(c_r1cs.num_constraints, c_r1cs.num_instance, c_r1cs.num_witness, c_r1cs.matrices())
            c_pk = ctx2.setup(h2, TRAPDOOR)
            gpu_proof = ctx2.prove(ctx2.pk_load(c_pk), h2, c_z, *r_s)
            ctx2.close()
            sample = f"1 proof of a 2^{CPU_SAMPLE_MAX_LOG_N}-2 constraint circuit of the same generator"
        t = time.perf_counter()
        cpu_proof, stage = oc.prove(cid, c_pk, c_r1cs, c_z, *r_s, fq_bytes)
        dt = time.perf_counter() - t
        if gpu_proof != cpu_proof:
            raise SystemExit(f"PARITY FAILURE: GPU proof ({world} rank(s)) differs from the CPU oracle")
        expected = oc.trapdoor_expected(cid, c_r1cs, TRAPDOOR, c_z, *r_s, fq_bytes)
        if expected != cpu_proof:
            raise SystemExit("PARITY FAILURE: proof differs from the trapdoor prediction")
        cpu_baseline = {"value": c_n / dt, "unit": "constraints/s", "cores": oc.threads(), "kind": "port",
                        "sample": sample + f": {dt:.1f} s, ark-equivalent C port of the reference's prover (MSM parallel over windows only as in "
                                           "ark 0.3.0); the GPU proof of the same (key, witness, r, s) is byte-identical and equals the trapdoor prediction",
                        "stage_s": {k: float(v) for k, v in zip(("pk_deserialize", "witness_map", "msm_g1", "msm_g2", "total"), stage)}}

    if rank == 0:
        line = {
            "metric": "groth16_constraints_per_sec", "value": value, "unit": "constraints/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_res / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u256-montgomery" if cid == 0 else "u384-montgomery", "data": "synthetic",
            "config": bench_config(args, world, r1cs.num_variables),
            "tables": table_info,
            "timing": "K proofs submitted AND collected between barrier + synchronize (two in flight: proof i+1's device work is enqueued "
                      "before the host part of proof i runs); wall clock = device clock of the region, max over ranks; per-stage CUDA "
                      "events on the launching streams are in stages_ms; latency_ms_one_proof_e2e is one proof alone",
            "e2e": {"value": e2e_value, "unit": "constraints/s", "h2d_bytes_per_step": int(z.nbytes + 64),
                    "d2h_bytes_per_step": int(256 + 4 * 2 * 72 * 128 + 2 * 72 * 256), "ms_per_step": 1e3 * t_e2e / args.steps},
            "gpu_launches": int(launches),
            "pipeline_depth": args.pipeline,
            "latency_ms_one_proof_e2e": latency_ms,
            "trait_shaped_call": trait_call,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "stages_ms": stage_res,
            "prep_s": round(prep_s, 1),
            "pk_bytes": pk_bytes,
        }
        sys.stdout.flush()
        os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)


if __name__ == "__main__":
    main()
