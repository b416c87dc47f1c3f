"""GPU: pb254_scalar_mul_chains (K13) on three workloads, next to the serial CPU chain and a config-2 proof.

    python tools/chain_bench.py [--reps 20] [--out r4_chains.json]

Workloads: G1 one chain of 1024 terms (a config-2 batch as one g1_msm), G1 64 chains of 128 terms (8192 terms, the
size of the reference's g1_msm_test), G2 1024 singleton chains from hash_to_g2_inputs rows (the cofactor clearings of
a config-3 batch). For each: the device time of every stage (ctx.timings(), CUDA events) and the host wall time of the
call, as medians over --reps calls after a warm-up; and the serial CPU chain on the same inputs (the oracle's
native_result term by term on one thread, as the generator loop runs). The outputs are compared with the serial chain.
A config-2 proof (G1, 1024 instances, 2^19 rows) of the chained batch is timed in the same run for proportion. The
card's name, power limit and maximum SM clock are read with nvidia-smi's read-only query.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from oracle import pyoracle as O  # noqa: E402
from plonky2_bn254_b200 import ffi, inputs as I, workloads as Wk  # noqa: E402

FW = {I.KIND_G1: 4, I.KIND_G2: 8}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"query": out[0], "gpu0": out[1]}


def limbs_to_words(limbs):
    l = np.asarray(limbs, dtype=np.uint64).reshape(-1, 4)
    return l[:, 0] | (l[:, 1] << np.uint64(16)) | (l[:, 2] << np.uint64(32)) | (l[:, 3] << np.uint64(48))


def serial_chains(kind, terms, starts, offsets):
    rows, sums = [], []
    for c in range(len(starts) - 1):
        acc = np.asarray(offsets[c], dtype=np.uint64)
        for i in range(int(starts[c]), int(starts[c + 1])):
            row = np.concatenate([terms[i], acc])
            rows.append(row)
            acc = limbs_to_words(O.native_result(kind, row))
        sums.append(acc)
    return np.array(rows, dtype=np.uint64), np.array(sums, dtype=np.uint64)


def workloads(ctx):
    tw = 4 + 2 * FW[I.KIND_G1]
    inp, _ = I.make_inputs(I.KIND_G1, 8192, I.config_seed(2))
    yield "g1_1chain_1024", I.KIND_G1, inp[:1024, :tw], np.array([0, 1024], dtype=np.uint64), inp[:1, tw:]
    yield ("g1_64chains_128", I.KIND_G1, inp[:, :tw], np.arange(0, 8193, 128, dtype=np.uint64), inp[:64, tw:])
    rng = np.random.default_rng(3)
    msgs = rng.integers(0, Wk.GOLDILOCKS_P, size=(1024, 8), dtype=np.uint64)
    g2, _, _ = Wk.hash_to_g2_inputs(msgs, ctx.poseidon_permute, seed=I.config_seed(3))
    yield "g2_1024_singletons", I.KIND_G2, g2[:, :20], np.arange(1025, dtype=np.uint64), g2[:, 20:]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="write the result as JSON (it is always printed)")
    a = ap.parse_args()
    O.build()
    ctx = ffi.Context(0)
    res = {"gpu": gpu_info(), "reps": a.reps, "workloads": {}}
    print(res["gpu"], flush=True)
    chained_g1 = None
    for name, kind, terms, starts, offsets in workloads(ctx):
        terms, offsets = np.ascontiguousarray(terms), np.ascontiguousarray(offsets)
        for _ in range(3):
            rows, sums = ctx.scalar_mul_chains(kind, terms, starts, offsets)
        walls, stages = [], {}
        for _ in range(a.reps):
            t = time.perf_counter()
            rows, sums = ctx.scalar_mul_chains(kind, terms, starts, offsets)
            walls.append((time.perf_counter() - t) * 1e3)
            for st, ms in ctx.timings():
                stages.setdefault(st, []).append(ms)
        t = time.perf_counter()
        want_rows, want_sums = serial_chains(kind, terms, starts, offsets)
        cpu_ms = (time.perf_counter() - t) * 1e3
        same = bool((rows == want_rows).all() and (sums == want_sums).all())
        dev = {st: statistics.median(v) for st, v in stages.items()}
        w = {"kind": "g1" if kind == I.KIND_G1 else "g2", "n_terms": int(terms.shape[0]), "n_chains": int(starts.size - 1),
             "device_ms_median": dev, "device_ms_total": sum(dev.values()),
             "host_wall_ms_median": statistics.median(walls), "host_wall_ms_min": min(walls),
             "serial_cpu_oracle_ms": cpu_ms, "equal_to_serial_oracle": same}
        res["workloads"][name] = w
        print(name, json.dumps(w), flush=True)
        if name == "g1_1chain_1024":
            chained_g1 = rows
    ts = np.arange(1024, dtype=np.uint64)
    for _ in range(2):
        pf = ctx.prove(I.KIND_G1, chained_g1, ts)
    prove_ms = []
    for _ in range(5):
        t = time.perf_counter()
        pf = ctx.prove(I.KIND_G1, chained_g1, ts)
        prove_ms.append((time.perf_counter() - t) * 1e3)
    res["config2_prove_of_chained_g1_batch"] = {"host_wall_ms_median": statistics.median(prove_ms),
                                                "verified": bool(ctx.L.verify(I.KIND_G1, pf.words(), chained_g1, ts))}
    g1 = res["workloads"]["g1_1chain_1024"]
    res["g1_1024_chain_share_of_proof"] = g1["host_wall_ms_median"] / statistics.median(prove_ms)
    print(json.dumps(res["config2_prove_of_chained_g1_batch"]), "share", res["g1_1024_chain_share_of_proof"], flush=True)
    print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
