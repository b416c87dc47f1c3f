"""GPU: pb254_hash_to_g2 (K14) at three batch sizes, next to the Python producer and a config-3 proof of the batch.

    python tools/hash_to_g2_bench.py [--reps 20] [--out r5_hash_to_g2.json]

For n in {1024, 16384, 131072} messages of 8 Goldilocks elements: the device time of every stage (ctx.timings(), CUDA
events) and the host wall time of the call, as medians over --reps calls after a warm-up. At n = 1024 the outputs are
compared with the Python producer (workloads.hash_to_g2_inputs with the oracle's Poseidon; hashes = the oracle's
native_result minus the offset), and the Python producer itself is timed with the device Poseidon and its fixed-base
table already built. A config-3 proof (G2, 1024 instances, 2^19 rows) of the same batch is timed in the same run for
proportion. The card's name, power limit and maximum SM clock are read with nvidia-smi's read-only query.
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

SIZES = (1024, 16384, 131072)
MSG_LEN = 8


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"query": out[0], "gpu0": out[1]}


def messages(n):
    rng = np.random.default_rng(n)
    return rng.integers(0, Wk.GOLDILOCKS_P, size=(n, MSG_LEN), dtype=np.uint64)


def oracle_permute(st):
    return np.stack([O.poseidon_permute(r) for r in np.asarray(st, dtype=np.uint64).reshape(-1, 12)])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="write the result as JSON (it is always printed)")
    a = ap.parse_args()
    O.build()
    ctx = ffi.Context(0)
    res = {"gpu": gpu_info(), "reps": a.reps, "msg_len": MSG_LEN, "sizes": {}}
    print(res["gpu"], flush=True)
    seed = I.config_seed(3)
    batch = None
    for n in SIZES:
        msgs = messages(n)
        for _ in range(3):
            inputs, hashes = ctx.hash_to_g2(msgs, seed)
        walls, stages = [], {}
        for _ in range(a.reps):
            t = time.perf_counter()
            inputs, hashes = ctx.hash_to_g2(msgs, seed)
            walls.append((time.perf_counter() - t) * 1e3)
            for st, ms in ctx.timings():
                stages.setdefault(st, []).append(ms)
        dev = {st: statistics.median(v) for st, v in stages.items()}
        w = {"n": n, "device_ms_median": dev, "device_ms_total": sum(dev.values()),
             "host_wall_ms_median": statistics.median(walls), "host_wall_ms_min": min(walls)}
        if n == SIZES[0]:
            batch = (msgs, inputs, hashes)
        res["sizes"][str(n)] = w
        print(n, json.dumps(w), flush=True)

    msgs, inputs, hashes = batch
    n = msgs.shape[0]
    rows, _, offs = Wk.hash_to_g2_inputs(msgs, oracle_permute, seed)
    native = np.array([O.native_result(I.KIND_G2, r) for r in rows])
    want_hashes = np.array([Wk._g2_words(h) for h in Wk.hash_to_g2_outputs(native, offs)], dtype=np.uint64)
    res["equal_to_python_at_1024"] = bool((inputs == rows).all() and (hashes == want_hashes).all())
    I.scalar_mul_gen(I.KIND_G2, 1)  # the Python fixed-base table is built once per process
    t = time.perf_counter()
    Wk.hash_to_g2_inputs(msgs, ctx.poseidon_permute, seed)
    res["python_producer_ms_at_1024"] = (time.perf_counter() - t) * 1e3
    print("equal", res["equal_to_python_at_1024"], "python ms", res["python_producer_ms_at_1024"], flush=True)

    ts = np.arange(n, dtype=np.uint64)
    for _ in range(2):
        pf = ctx.prove(I.KIND_G2, inputs, ts)
    prove_ms = []
    for _ in range(5):
        t = time.perf_counter()
        pf = ctx.prove(I.KIND_G2, inputs, ts)
        prove_ms.append((time.perf_counter() - t) * 1e3)
    res["config3_prove_of_batch"] = {"host_wall_ms_median": statistics.median(prove_ms),
                                     "verified": bool(ctx.L.verify(I.KIND_G2, pf.words(), inputs, ts))}
    res["h2g2_1024_share_of_proof"] = res["sizes"]["1024"]["host_wall_ms_median"] / statistics.median(prove_ms)
    print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
