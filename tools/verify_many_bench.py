"""GPU: N sequential pb254_verify_device calls against one pb254_verify_many_device call on the same N proofs.

    python tools/verify_many_bench.py [--reps 5] [--out profiles/r8_verify_many.json]

Workloads (proofs made by ffi.prove_many on one context, seeded): G1 x 128 instances (2^16 rows) at N = 1, 8, 32, 64;
G2 x 128 at N = 1, 8, 32; G1 x 1024 (config 2, 2^19 rows) at N = 1, 8. For each workload and N the two ways are called
alternately in one process, one warm-up and --reps timed calls each; every call ends in a stream synchronise, so the
host wall time around it is the call time. Reported: the medians, the device stage times of verify_many ("verify
native ctl", "verify merkle"; CUDA events), its host remainder (wall minus the stages: threads, transcripts, quotient
identities, the upload and the FRI folds), and that both ways accepted every proof. At N = 1 pb254_verify (the host
verifier) is timed too. The card's name and power limit are read with nvidia-smi's read-only query.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from plonky2_bn254_b200 import ffi, inputs as I  # noqa: E402
from verify_bench import gpu_info  # noqa: E402

WORKLOADS = [("g1x128", I.KIND_G1, 128, (1, 8, 32, 64)), ("g2x128", I.KIND_G2, 128, (1, 8, 32)),
             ("g1x1024", I.KIND_G1, 1024, (1, 8))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the result as JSON (it is always printed)")
    a = ap.parse_args()
    ctx = ffi.Context(0)
    res = {"gpu": gpu_info(), "reps": a.reps, "workloads": {}}
    print(res["gpu"], flush=True)
    for name, kind, n, ns in WORKLOADS:
        batches = [I.make_inputs(kind, n, I.config_seed(900 + 10 * kind + b)) for b in range(max(ns))]
        t = time.perf_counter()
        proofs = [p.words() for p in ffi.prove_many([ctx], kind, batches)]
        prove_ms = (time.perf_counter() - t) * 1e3
        rows = {"kind": I.KIND_NAMES[kind], "instances": n, "degree_bits": int(proofs[0][2]),
                "proof_words": int(proofs[0].size), "prove_many_ms": prove_ms, "by_n": {}}
        for N in ns:
            calls = {"sequential": lambda: all(ctx.verify(kind, proofs[b], *batches[b]) for b in range(N)),
                     "many": lambda: ctx.verify_many(kind, proofs[:N], batches[:N]) == [None] * N}
            if N == 1:
                calls["host"] = lambda: ctx.L.verify(kind, proofs[0], *batches[0])
            accepted = {k: bool(f()) for k, f in calls.items()}  # warm-up
            walls, stages = {k: [] for k in calls}, {}
            for _ in range(a.reps):
                for k, f in calls.items():
                    t = time.perf_counter()
                    accepted[k] &= bool(f())
                    walls[k].append((time.perf_counter() - t) * 1e3)
                    if k == "many":
                        for st, ms in ctx.timings():
                            stages.setdefault(st, []).append(ms)
            med = {k: statistics.median(v) for k, v in walls.items()}
            dev = {st: statistics.median(v) for st, v in stages.items()}
            r = {"sequential_verify_ms_median": med["sequential"], "verify_many_ms_median": med["many"],
                 "sequential_verify_ms_all": walls["sequential"], "verify_many_ms_all": walls["many"],
                 "verify_many_stage_ms_median": dev,
                 "verify_many_host_remainder_ms": med["many"] - sum(dev.values()),
                 "speedup": med["sequential"] / med["many"], "all_accepted": all(accepted.values())}
            if N == 1:
                r["pb254_verify_ms_median"] = med["host"]
                r["pb254_verify_ms_all"] = walls["host"]
            rows["by_n"][N] = r
            print(name, N, json.dumps(r), flush=True)
        res["workloads"][name] = rows
    print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
