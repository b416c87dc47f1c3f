"""GPU: pb254_verify (host) against pb254_verify_device (K15) on one proof per BASELINE config.

    python tools/verify_bench.py [--reps 5] [--config5] [--out r6_verify.json]

Configs: 1 (G1 x 1, 2^16 rows), 2 (G1 x 1024, 2^19 rows), 3 (G2 x 1024, 2^19 rows), 4b (fq_exp x 4096, 2^21 rows,
rate_bits 3 and 28 query rounds, as bench.py sets it) and with --config5 5 (G1 x 8192, 2^22 rows, one GPU). Each config
proves one seeded batch, then calls Library.verify and Context.verify on it alternately, one warm-up and --reps timed
calls each, in the same process. Reported per config: the medians of the host wall times, the device stage times of
pb254_verify_device ("verify native ctl", "verify merkle"; CUDA events), the host remainder of the device call (wall
minus the device stages: parsing, transcript, quotient identity at zeta, uploads and FRI folds), the proof time, and
that both verifiers accepted. The card's name and power limit are read with nvidia-smi's read-only query.
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

from plonky2_bn254_b200 import ffi, inputs as I  # noqa: E402


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()
    return {"query": out[0], "gpu0": out[1]}


def configs(lib, with_config5):
    yield "1", I.KIND_G1, 1, 1, None
    yield "2", I.KIND_G1, 1024, 2, None
    yield "3", I.KIND_G2, 1024, 3, None
    cfg = lib.standard_fast_config()
    cfg.rate_bits, cfg.num_query_rounds = 3, 28
    yield "4b", I.KIND_FQ, 4096, 4, cfg
    if with_config5:
        yield "5", I.KIND_G1, 8192, 5, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--config5", action="store_true")
    ap.add_argument("--out", default=None, help="write the result as JSON (it is always printed)")
    a = ap.parse_args()
    ctx = ffi.Context(0)
    res = {"gpu": gpu_info(), "reps": a.reps, "configs": {}}
    print(res["gpu"], flush=True)
    for name, kind, n, seed, cfg in configs(ctx.L, a.config5):
        inp, ts = I.make_inputs(kind, n, I.config_seed(seed))
        t = time.perf_counter()
        w = ctx.prove(kind, inp, ts, config=cfg).words()
        prove_ms = (time.perf_counter() - t) * 1e3
        calls = {"host": lambda: ctx.L.verify(kind, w, inp, ts, config=cfg),
                 "device": lambda: ctx.verify(kind, w, inp, ts, config=cfg)}
        accepted = {k: bool(f()) for k, f in calls.items()}  # warm-up
        walls, stages = {"host": [], "device": []}, {}
        for _ in range(a.reps):
            for k, f in calls.items():
                t = time.perf_counter()
                accepted[k] &= bool(f())
                walls[k].append((time.perf_counter() - t) * 1e3)
                if k == "device":
                    for st, ms in ctx.timings():
                        stages.setdefault(st, []).append(ms)
        host_ms, dev_ms = statistics.median(walls["host"]), statistics.median(walls["device"])
        dev_stages = {st: statistics.median(v) for st, v in stages.items()}
        r = {"kind": I.KIND_NAMES[kind], "instances": n, "degree_bits": int(w[2]), "rate_bits": int(w[3]),
             "query_rounds": int(w[6]), "proof_words": int(w.size), "prove_ms_first_call": prove_ms,
             "pb254_verify_ms_median": host_ms, "pb254_verify_device_ms_median": dev_ms,
             "pb254_verify_ms_all": walls["host"], "pb254_verify_device_ms_all": walls["device"],
             "device_stage_ms_median": dev_stages,
             "device_call_host_remainder_ms": dev_ms - sum(dev_stages.values()),
             "speedup": host_ms / dev_ms, "both_accepted": accepted["host"] and accepted["device"]}
        res["configs"][name] = r
        print(name, json.dumps(r), flush=True)
    print(json.dumps(res), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
