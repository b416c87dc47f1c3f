#!/usr/bin/env python
"""Headline benchmark: G1 scalar-mul STARK proofs/sec (BASELINE.json `metric`), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--instances 1024] [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch: generate_trace + prove of `--instances` G1
scalar-muls in ONE trace (default 1024 => 2^19 rows x 781 columns = BASELINE.json configs[1], SURVEY.md
section 8d "config 2"), StarkConfig::standard_fast_config(). Synthetic inputs: SplitMix64-seeded random
256-bit scalars and random subgroup points (plonky2_bn254_b200/inputs.py), a different batch per rank.

  value  proofs/s with the work items already resident in HBM (pb254_prove_dev), device-timed
  e2e    proofs/s through the host-buffer C-ABI call pb254_prove (pinned host inputs -> H2D, proof -> D2H
         and a host checksum of the proof bytes inside the timed region)
  roofline     the dominant kernel (Merkle leaf hashing + inner levels, K4+K5) against measured HBM peak
               with SURVEY.md 8(d)'s algorithmic bytes; `ntt` carries the same for the LDE kernels (K3)
  cpu_baseline the CPU oracle (a restatement of the reference prover; the Rust crate cannot be built
               offline) on a bounded sample, timed on this box's host cores

  other_configs    BASELINE configs 3 (G2 x 1024) and 4 (fq_exp x 4096, blow-up 8), measured in the same run
  pipelined        pb254_prove_many: a stream of proofs through two contexts of the same GPU
  oversized_trace  N > 1 only: BASELINE config 5, ONE proof of 2^22 rows across all N GPUs (pb254_prove_sharded:
                   column-sharded LDE, NCCL all-to-all, row-block hashing / quotient / FRI combination)

N > 1 (torchrun): independent proof batches per GPU (replicas, SURVEY.md 8e) - no data-path collective for the
headline value; the NCCL process group is used for the barrier, the max-over-ranks time and the oversized proof.

`--impl reference` times the reference's CPU algorithm (the oracle port, all host threads) on a bounded
sample of the same workload; this and the cpu_baseline leg are the only places bench.py executes oracle/.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "g1_scalar_mul_stark_proofs_per_sec"
UNIT = "proofs/s"
KIND_G1 = 0


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_metrics():
    """Numbers that only a profiler can give (DRAM bytes per launch, executed instructions, pipe utilisation), as
    tools/make_profiles.py extracted them from the ncu captures committed under profiles/; the file carries the
    commit and date of the capture. Nothing of this kind is typed into bench.py by hand."""
    try:
        with open(os.path.join(ROOT, "profiles", "current_metrics.json")) as f:
            name = json.load(f)["file"]
        with open(os.path.join(ROOT, "profiles", name)) as f:
            m = json.load(f)
        m["_file"] = "profiles/" + name
        return m
    except Exception:
        return None


def leaf_hash_profile(m, perms_per_launch):
    """The largest captured leaf-hash launch (the trace tree of a config-2 proof) of the metrics file."""
    if not m:
        return None
    best, kname, pipes = None, None, {}
    for k, v in m.get("kernels", {}).items():
        if "leaf_hash" not in k:
            continue
        if v.get("issue_active") is not None:  # the per-kernel table (section capture) of the same proof
            pipes = {x: v.get(x) for x in ("issue_active", "alu_pipe", "fma_heavy_pipe", "warps_active", "registers")}
        for c in v.get("full_captures", []):
            if c.get("dram_bytes") and (best is None or c["dram_bytes"] > best["dram_bytes"]):
                best, kname = dict(c), k
    if best:
        best.update(pipes)
    if not best:
        return None
    out = {"source": f"{m['_file']} (commit {m.get('commit')}, {m.get('date')}): ncu --set full capture of {kname}, "
                     f"grid {best.get('grid')}",
           "dram_bytes_per_launch": best["dram_bytes"], "ms_under_ncu": best["ms"]}
    if best.get("warp_instructions"):
        ti = 32.0 * best["warp_instructions"] / perms_per_launch
        out.update({"thread_instructions_per_permutation": ti,
                    "issue_peak_gperm_per_s": 148 * 128 * 1.965e9 / ti / 1e9})
    for x, y in (("issue_active", "issue_active"), ("alu_pipe", "alu_pipe_busy"), ("fma_heavy_pipe", "fma_heavy_pipe_busy"),
                 ("warps_active", "warps_active"), ("registers", "registers_per_thread")):
        if best.get(x) is not None:
            out[y] = best[x]
    return out


def algorithmic_bytes(W, A, Q, n, rate_bits, cap_height):
    """SURVEY.md 8(d): bytes_ntt(C,n,b) = 8 C n (2 + b); bytes_merkle(C,n,b) = 8 C n b + 32 (2 n b - 2^cap)."""
    b = 1 << rate_bits
    ntt = sum(8 * c * n * (2 + b) for c in (W, A)) + 8 * Q * n * (1 + b)  # quotient chunks come as coefficients
    merkle = sum(8 * c * n * b + 32 * (2 * n * b - (1 << cap_height)) for c in (W, A, Q))
    return ntt, merkle


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.sm_max = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake_slowdown",
        }
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(sm)}


def physical_device_index(local_index):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_index])
        except Exception:
            return local_index
    return local_index


# ------------------------------------------------------------------------------------------------
_CPU_INPUTS = {}


def cpu_sample(sample_instances, repeats=1):
    """One oracle proof (trace generation + prove) of `sample_instances` G1 scalar-muls; seconds (best).
    Uses every host core (torchrun exports OMP_NUM_THREADS=1, which would otherwise throttle the baseline)."""
    from oracle import pyoracle as O
    from plonky2_bn254_b200 import inputs as I
    O.set_num_threads(os.cpu_count() or 1)
    if sample_instances not in _CPU_INPUTS:  # workload generation is not part of the timed sample
        _CPU_INPUTS[sample_instances] = I.make_inputs(KIND_G1, sample_instances, I.config_seed(1))
    inp, ts = _CPU_INPUTS[sample_instances]
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        pf, t_trace, t_prove = O.prove_inputs(KIND_G1, inp, ts)
        dt = time.perf_counter() - t0
        del pf
        best = dt if best is None else min(best, dt)
    return best, O.num_threads()


def rows_for(instances):
    return max(1 << 16, 1 << (instances * 512 - 1).bit_length())


def cpu_baseline(instances, sample_instances):
    """The CPU oracle on THIS workload, measured, not extrapolated: one full proof (generate_trace + prove of
    `instances` scalar-muls, all host cores). The 1/8-size sample the reference arm steps on is timed beside it so
    that the scale factor between the two is a measurement as well."""
    t_full, threads = cpu_sample(instances)
    out = {
        "value": 1.0 / t_full, "unit": UNIT, "cores": threads, "kind": "port",
        "sample": (f"ONE full oracle proof of the workload itself (generate_trace + prove, {instances} G1 scalar-muls, "
                   f"{rows_for(instances)} rows) took {t_full:.2f} s on {threads} threads; value = 1 / that time. "
                   f"The Rust reference cannot be compiled offline (no cargo, un-vendored git dependencies): the "
                   f"oracle is a C++/OpenMP restatement of the same algorithm"),
        "sample_seconds": t_full,
        "scalar_muls_per_s": instances / t_full,
    }
    if sample_instances < instances:
        t_s, _ = cpu_sample(sample_instances)
        frac = rows_for(sample_instances) / rows_for(instances)
        out["reduced_sample"] = {
            "instances": sample_instances, "trace_rows": rows_for(sample_instances), "seconds": t_s,
            "fraction_of_workload_rows": frac,
            "full_over_sample_time": t_full / t_s, "rows_ratio": 1.0 / frac,
            "note": "the reference arm (--impl reference) steps on this sample; full_over_sample_time is the measured "
                    "cost ratio against the rows ratio it assumes"}
    return out


def run_reference(args, rank, world):
    """The reference's CPU algorithm (oracle port, every host thread) on a bounded sample per step.

    A step proves `sample` of the workload's `instances` scalar-muls (a 2^16-row trace, 1/8 of the 2^19 rows):
    ms_per_step is the TRUE time of such a step and value = (fraction of one workload proof done per step) / step
    time, so steps x ms_per_step is the real timed region. One full workload proof is timed before the steps
    (outside the timed region) and reported as `full_workload_check`, which pins the scale factor by measurement."""
    if rank != 0:
        return
    sample = min(args.cpu_sample_instances, args.instances)
    n_full, n_samp = rows_for(args.instances), rows_for(sample)
    frac = n_samp / n_full
    full_check = None
    if not args.no_full_check and sample < args.instances:
        t_full, _ = cpu_sample(args.instances)
        full_check = {"seconds": t_full, "proofs_per_s": 1.0 / t_full,
                      "what": f"one full oracle proof of {args.instances} scalar-muls ({n_full} rows), timed once "
                              f"before the steps"}
    for _ in range(args.warmup):
        cpu_sample(sample)
    t0 = time.perf_counter()
    threads = 1
    for _ in range(args.steps):
        _, threads = cpu_sample(sample)
    dt = (time.perf_counter() - t0) / args.steps
    value = frac / dt
    if full_check:
        full_check["value_over_full_workload_rate"] = value / full_check["proofs_per_s"]
    cfg = workload_config(args)
    cfg["reference_step"] = {
        "instances_per_step": sample, "trace_rows_per_step": n_samp, "fraction_of_workload_per_step": frac,
        "note": "each timed step is one CPU proof of a bounded sample of the workload (same columns, same "
                "StarkConfig, 1/8 of the rows); value counts the fraction of a workload proof completed per second"}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {
            "value": value, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": (f"each step = one CPU-oracle proof of {sample} G1 scalar-muls ({n_samp} rows = {frac:g} of the "
                       f"workload's {n_full} rows) in {dt:.2f} s; value = {frac:g} / step time. The Rust reference "
                       f"cannot be compiled offline (no cargo, un-vendored git dependencies); the oracle is a "
                       f"C++/OpenMP restatement of the same algorithm.")},
        "full_workload_check": full_check,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(args):
    n = max(1 << 16, 1 << (args.instances * 512 - 1).bit_length())
    return {
        "workload": f"batched G1 scalar-mul STARK, {args.instances} scalar-muls in one trace "
                    f"({n} rows x 781 columns), generate_trace + prove, StarkConfig::standard_fast_config",
        "instances_per_proof": args.instances, "trace_rows": n, "trace_columns": 781, "aux_columns": 456,
        "rate_bits": 1, "num_query_rounds": 84, "pow_bits": 16,
        "parallelism": f"replicas x{args.gpus} (independent proof batches per GPU, no collective)",
        "l2_policy": "inputs larger than L2: every kernel streams a >= 3 GiB trace / LDE matrix (L2 = 126 MB)",
    }


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    from plonky2_bn254_b200 import ffi, inputs as I

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the prover has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist = dist_mod

    stream = torch.cuda.Stream(device=local_rank)
    ctx = ffi.Context(local_rank, stream=stream.cuda_stream)
    lib = ctx.L

    # a different batch per rank and per step (3 distinct batches, cycled)
    nb = 3
    batches = [I.make_inputs(KIND_G1, args.instances, I.config_seed(2) + 1000 * rank + b) for b in range(nb)]
    pinned = [(torch.from_numpy(inp.view(np.int64)).pin_memory(), torch.from_numpy(ts.view(np.int64)).pin_memory())
              for inp, ts in batches]
    on_dev = [(a.to(f"cuda:{local_rank}"), b.to(f"cuda:{local_rank}")) for a, b in pinned]
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local_rank}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_dev(i):
        a, b = on_dev[i % nb]
        pf = ctx.prove_dev(KIND_G1, a.data_ptr(), b.data_ptr(), args.instances)
        return pf

    def step_host(i):
        a, b = pinned[i % nb]
        pf = ctx.prove(KIND_G1, a.numpy().view(np.uint64).reshape(args.instances, 20), b.numpy().view(np.uint64))
        w = pf.words()  # the step's result on the host: the serialized proof
        return pf, zlib.crc32(w.tobytes()), w.size * 8

    # ---- warm-up -----------------------------------------------------------------------------
    for i in range(args.warmup):
        step_dev(i).close()
    for i in range(min(args.warmup, 3)):
        step_host(i)[0].close()

    # ---- value: inputs resident in HBM ---------------------------------------------------------
    sampler = ClockSampler(physical_device_index(local_rank))
    stage_ms: dict = {}
    launches0 = lib.launch_count()
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    last = None
    for i in range(args.steps):
        pf = step_dev(i)
        for name, ms in ctx.timings():
            stage_ms[name] = stage_ms.get(name, 0.0) + ms
        if i + 1 < args.steps:
            pf.close()
        else:
            last = pf  # read back after the timed region
    ev1.record(stream)
    barrier()
    dev_s = max_over_ranks(ev0.elapsed_time(ev1) * 1e-3)
    launches = lib.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "proof_words": u64_as_f64_halves(last.words()),
            "results": last.results().reshape(args.instances, -1).astype(np.float64)})
    last.close()

    # ---- e2e: host buffers through the C ABI ---------------------------------------------------
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    d2h = 0
    for i in range(args.steps):
        pf, _crc, nbytes = step_host(i)
        d2h = nbytes
        pf.close()
    e1.record(stream)
    barrier()
    # every step ends with a stream synchronise inside the C-ABI call, so the event interval on the
    # context's stream covers the host work (transcript, proof assembly, checksum) as well
    e2e_s = max_over_ranks(e0.elapsed_time(e1) * 1e-3)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    # ---- a stream of proofs through two contexts of the same GPU (pb254_prove_many) ----------------
    pipelined = None
    if not args.no_pipelined:
        stream2 = torch.cuda.Stream(device=local_rank)
        ctx2 = ffi.Context(local_rank, stream=stream2.cuda_stream)
        many = [batches[i % nb] for i in range(2 * args.steps)]
        for pf in ffi.prove_many([ctx, ctx2], KIND_G1, many[:2]):  # warm-up (second workspace, lazy module loads)
            pf.close()
        barrier()
        t0 = time.perf_counter()
        pfs = ffi.prove_many([ctx, ctx2], KIND_G1, many)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        for pf in pfs:
            pf.close()
        ctx2.close()
        pipelined = {"what": "pb254_prove_many: independent proofs round-robin over two contexts (streams, workspaces, host "
                             "threads) of one GPU, host input buffers, proofs returned to the host; wall clock",
                     "contexts": 2, "proofs": len(many), "proofs_per_s": world * len(many) / dt,
                     "ms_per_proof": dt / len(many) * 1e3}

    # ---- BASELINE.json configs 3 and 4 (secondary keys, same run, same replica layout) -------------
    other = {}
    if not args.no_other_configs:
        cases = [("config3_g2_x1024", 1, 1024, None,
                  "G2 scalar-mul STARK, 1024 scalar-muls in one trace (2^19 rows x 1295 columns), standard_fast_config"),
                 ("config4_fq_exp_x4096_blowup8", 2, 4096, (3, 28),
                  "fq_exp STARK, 4096 exponentiations in one trace (2^21 rows x 427 columns), rate_bits 3, 28 query rounds")]
        for key, kind, k, rb, what in cases:
            inp, ts = I.make_inputs(kind, k, I.config_seed(3 + kind) + 1000 * rank)
            d_in = torch.from_numpy(inp.view(np.int64)).to(f"cuda:{local_rank}")
            d_ts = torch.from_numpy(ts.view(np.int64)).to(f"cuda:{local_rank}")
            cfg = None
            if rb:
                cfg = lib.standard_fast_config()
                cfg.rate_bits, cfg.num_query_rounds = rb
            ctx.prove_dev(kind, d_in.data_ptr(), d_ts.data_ptr(), k, config=cfg).close()  # warm-up
            st: dict = {}
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(stream)
            for _ in range(args.other_steps):
                pf = ctx.prove_dev(kind, d_in.data_ptr(), d_ts.data_ptr(), k, config=cfg)
                for name, ms in ctx.timings():
                    st[name] = st.get(name, 0.0) + ms
                pf.close()
            s1.record(stream)
            barrier()
            sec = max_over_ranks(s0.elapsed_time(s1) * 1e-3)
            Wk, Ak = lib.trace_width(kind), lib.num_aux(kind, 2)
            nk = lib.trace_rows(k, 1 << 16)
            Nk = nk << (rb[0] if rb else 1)
            mk_ms = (st.get("merkle trace", 0) + st.get("merkle aux", 0)) / args.other_steps
            perms = sum(((c + 7) // 8) * Nk for c in (Wk, Ak)) + 2 * (Nk - 16)
            other[key] = {"workload": what, "proofs_per_s": world * args.other_steps / sec,
                          "ms_per_proof": sec / args.other_steps * 1e3, "steps": args.other_steps, "warmup": 1,
                          "instances_per_proof": k, "instances_per_s": world * args.other_steps * k / sec,
                          "trace_rows": nk, "trace_columns": Wk, "aux_columns": Ak, "lde_rows": Nk,
                          "poseidon_gperm_per_s": perms / (mk_ms * 1e-3) / 1e9 if mk_ms > 0 else None,
                          "stage_ms": {a: round(b / args.other_steps, 3) for a, b in st.items()}}
            del d_in, d_ts

    # ---- BASELINE.json config 5: ONE oversized trace proved across all N ranks (SURVEY.md 8e) --------
    oversized = None
    if dist is not None and not args.no_oversized:
        import hashlib
        from plonky2_bn254_b200 import dist as D
        for inst in (args.oversized_instances, args.oversized_instances // 2):
            try:
                o_inp, o_ts = I.make_inputs(KIND_G1, inst, I.config_seed(5))
                pf, coll = D.prove_sharded(ctx, dist, KIND_G1, o_inp, o_ts, f"cuda:{local_rank}", torch_stream=stream)
                pf.close()
                best, o_stage = None, None
                for _ in range(args.other_steps):
                    barrier()
                    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    s0.record(stream)
                    pf, coll = D.prove_sharded(ctx, dist, KIND_G1, o_inp, o_ts, f"cuda:{local_rank}", torch_stream=stream)
                    s1.record(stream)
                    barrier()
                    ms = max_over_ranks(s0.elapsed_time(s1))
                    if best is None or ms < best:
                        best, o_stage = ms, ctx.timings()
                    sha = hashlib.sha256(pf.words().tobytes()).hexdigest()
                    pf.close()
                shas = [None] * world
                dist.all_gather_object(shas, sha)
                ex = sum(v for k, v in o_stage if "exchange" in k)
                oversized = {
                    "workload": f"ONE G1 proof of {inst} scalar-muls ({lib.trace_rows(inst, 1 << 16)} rows x 781 columns) "
                                f"across {world} GPUs: column-sharded LDE, NCCL all-to-all into row blocks, row-block "
                                f"hashing / quotient / FRI combination, replicated transcript (pb254_prove_sharded)",
                    "instances": inst, "trace_rows": lib.trace_rows(inst, 1 << 16), "n_gpus": world,
                    "ms_per_proof": best, "proofs_per_s": 1e3 / best, "scalar_muls_per_s": inst * 1e3 / best,
                    "steps": args.other_steps, "warmup": 1, "identical_on_all_ranks": len(set(shas)) == 1,
                    "all_to_all_bytes_sent_per_rank": coll.bytes_all_to_all,
                    "all_gather_bytes_received_per_rank": coll.bytes_all_gather, "collective_calls": coll.calls,
                    "exchange_ms": ex,
                    "all_to_all_gb_s_per_rank": coll.bytes_all_to_all / (ex * 1e-3) / 1e9 if ex > 0 else None,
                    "stage_ms": {k: round(v, 3) for k, v in o_stage}}
                break
            except ffi.Pb254Error as e:  # the same on every rank (sizes are identical): try half the trace
                oversized = {"error": str(e), "instances": inst}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    W, A, Q = lib.trace_width(KIND_G1), lib.num_aux(KIND_G1, 2), 4
    n = lib.trace_rows(args.instances, 1 << 16)
    ntt_bytes, merkle_bytes = algorithmic_bytes(W, A, Q, n, 1, 4)
    per = {k: v / args.steps for k, v in stage_ms.items()}
    merkle_ms = per.get("merkle trace", 0) + per.get("merkle aux", 0)
    ntt_ms = per.get("lde trace", 0) + per.get("lde aux", 0)
    # "lde+merkle quotient" is one stage (4 columns); attribute it by its byte share
    qstage = per.get("lde+merkle quotient", 0.0)
    q_ntt_b, q_mk_b = 8 * Q * n * 3, 8 * Q * n * 2 + 32 * (4 * n - 16)
    merkle_ms += qstage * q_mk_b / (q_ntt_b + q_mk_b)
    ntt_ms += qstage * q_ntt_b / (q_ntt_b + q_mk_b)
    peak, peak_src = peaks()
    N = 2 * n
    leaf_perms = sum(((c + 7) // 8) * N for c in (W, A)) + 3 * (N - 16)

    def roof(bytes_, ms):
        ach = bytes_ / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None}

    # dominant kernel: k_leaf_hash (+ the small k_level launches) of the TRACE tree, one launch group per proof
    lead_bytes = 8 * W * N + 32 * (2 * N - 16)
    lead_ms = per.get("merkle trace", 0.0)
    lead_perms = ((W + 7) // 8) * N + (N - 16)
    roofline = roof(lead_bytes, lead_ms)
    prof = leaf_hash_profile(profile_metrics(), ((W + 7) // 8) * N) if args.instances == 1024 else None
    roofline.update({
        "kernel": "merkle leaf hash + inner levels, trace tree (781 columns x 2^20 LDE rows, Poseidon-Goldilocks, K4+K5)",
        "peak_source": peak_src, "algorithmic_bytes_per_launch": lead_bytes, "ms_per_launch": lead_ms,
        "share_of_step": lead_ms / (dev_s / args.steps * 1e3),
        # dram__bytes_read.sum + dram__bytes_write.sum of this launch from the committed ncu --set full capture
        "traffic": prof["dram_bytes_per_launch"] if prof else None,
        "poseidon_permutations_per_launch": lead_perms,
        "poseidon_gperm_per_s": lead_perms / (lead_ms * 1e-3) / 1e9 if lead_ms > 0 else 0.0,
        "int_pipe": prof,
        "all_trees": {"algorithmic_bytes_per_proof": merkle_bytes, "ms_per_proof": merkle_ms,
                      "achieved_gb_s": merkle_bytes / (merkle_ms * 1e-3) / 1e9 if merkle_ms > 0 else 0.0,
                      "poseidon_permutations_per_proof": leaf_perms},
        "note": "instruction-issue bound, not HBM bound (a Poseidon permutation costs ~2 x 10^4 integer instructions per "
                "64 absorbed bytes against a machine balance of 5.7 instructions per byte); the HBM fraction is "
                "reported because the contract asks for it, `int_pipe` (from the committed ncu capture) and DESIGN.md "
                "4.1 have the integer-pipe roofline",
    })
    ntt = roof(ntt_bytes, ntt_ms)
    ntt.update({"kernel": "coset LDE (iNTT + coset NTT, K3) of trace / aux / quotient columns",
                "algorithmic_bytes_per_proof": ntt_bytes, "ms_per_proof": ntt_ms,
                "share_of_step": ntt_ms / (dev_s / args.steps * 1e3), "peak_source": peak_src})

    line = {
        "metric": METRIC, "value": world * args.steps / dev_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_s / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args),
        "scalar_muls_per_s": world * args.steps * args.instances / dev_s,
        "e2e": {"value": world * args.steps / e2e_s, "unit": UNIT,
                "h2d_bytes_per_step": args.instances * 21 * 8, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "clocks": sampler.result(),
        "roofline": roofline,
        "ntt": ntt,
        "stage_ms": {k: round(v, 3) for k, v in per.items()},
    }
    if pipelined:
        line["pipelined"] = pipelined
    if other:
        line["other_configs"] = other
    if oversized:
        line["oversized_trace"] = oversized
    if not args.no_cpu_baseline and world == 1:  # rank 0 at N = 1 only
        line["cpu_baseline"] = cpu_baseline(args.instances, args.cpu_sample_instances)
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def u64_as_f64_halves(words):
    """uint64 words -> (n, 2) float64 [low 32 bits, high 32 bits]: a Goldilocks element does not fit float64's
    53-bit mantissa, its two halves do, so the file holds the words exactly."""
    import numpy as np
    w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1)
    return np.stack([w & np.uint64(0xFFFFFFFF), w >> np.uint64(32)], axis=1).astype(np.float64)


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy, so that two builds can be compared output for output."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: outputs of {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_REAL_STDOUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries (NCCL prints its version banner, torchrun its OMP note)
    write to fd 1 on their own, so fd 1 is pointed at stderr for the whole run and the JSON line goes to a saved
    copy of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=1024, help="G1 scalar-muls per proof (1024 = config 2)")
    ap.add_argument("--cpu-sample-instances", type=int, default=128)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the secondary measurements of BASELINE configs 3 (G2 x 1024) and 4 (fq_exp x 4096, blow-up 8)")
    ap.add_argument("--other-steps", type=int, default=2)
    ap.add_argument("--no-pipelined", action="store_true", help="skip the two-context pb254_prove_many measurement")
    ap.add_argument("--no-oversized", action="store_true",
                    help="N > 1: skip the one-proof-across-all-GPUs measurement (BASELINE config 5)")
    ap.add_argument("--oversized-instances", type=int, default=8192, help="8192 G1 scalar-muls = 2^22 rows (config 5)")
    ap.add_argument("--no-full-check", action="store_true",
                    help="reference arm: skip the one full-workload proof timed before the steps")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float64: proof_words "
                         "(n x 2: low and high 32 bits of each u64 proof word) and results (instances x 16-bit limbs "
                         "of the native outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run on this node
        import subprocess
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517"),
               os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
