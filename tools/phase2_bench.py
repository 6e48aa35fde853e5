#!/usr/bin/env python3
"""Times phase 2 of the ceremony (SURVEY.md config C5: MPCParameters::contribute / verify on the H and L queries) on
BLS12-377 with H = 2^20 - 1 and L = 2^20 elements in compressed host buffers, three ways:

  whole       ss_phase2_contribute / ss_phase2_verification on the first device
  sharded     the same calls with every visible device selected (ss_init), each query split across them
  primitives  the composition a caller needs without the phase-2 calls: contribute = transcode -> batch_mul ->
              transcode per query (delta^-1 from the host) plus batch_mul of delta_g1 / delta_g2; verify =
              check_subgroup of both `after` queries + merge_pairs per query + check_same_ratio per query

Each variant is warmed up once and timed over --reps calls (host clock around calls that return after a device
synchronise).  Contribute works in place, so repeated calls keep multiplying the same buffers; the cost is the same.

    python tools/phase2_bench.py --out results.json
"""
import argparse
import hashlib
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import pyref as R  # noqa: E402
import snark_setup_b200 as S  # noqa: E402
from snark_setup_b200 import ffi  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines() if out else ["unknown"]
    except Exception as e:  # noqa: BLE001
        return ["unknown (%s)" % e]


def timed(fn, reps):
    fn()  # warm-up: module load, lane allocation
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return {"call_ms": [round(1e3 * t, 1) for t in ts], "best_ms": round(1e3 * min(ts), 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", type=int, default=20, help="L = 2^log2 elements, H = 2^log2 - 1")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    cv, cid = R.BLS12_377, S.BLS12_377
    g1, g2 = cv.g1, cv.g2
    rng = random.Random(2025)
    n_l = 1 << a.log2
    n_h = n_l - 1
    tau, d_prev, delta = (rng.randrange(2, cv.r) for _ in range(3))
    inv = pow(delta, -1, cv.r)
    seed = hashlib.blake2b(b"phase2 bench", digest_size=32).digest()
    gen = g1.encode(g1.gen, True)
    # before: powers of a random tau (unstructured points), compressed as phase-2 files are written
    hb = S.apply_powers(cid, S.G1, gen * n_h, True, S.CHECK_NO, True, n_h, tau=tau, first_power=1)
    lb = S.apply_powers(cid, S.G1, gen * n_l, True, S.CHECK_NO, True, n_l, tau=tau, first_power=7)
    d1b = g1.encode(g1.mul(g1.gen, d_prev), True)
    d2b = g2.encode(g2.mul(g2.gen, d_prev), True)
    ha, la, d1a, d2a = bytearray(hb), bytearray(lb), bytearray(d1b), bytearray(d2b)
    S.phase2_contribute(cid, delta, ha, la, True, S.CHECK_NO, d1a, d2a)
    ha, la, d1a, d2a = bytes(ha), bytes(la), bytes(d1a), bytes(d2a)
    S.phase2_verification(cid, hb, ha, lb, la, True, d1a, d2b, d2a, seed=seed)  # the round is valid

    devices = S.lib().ss_device_count()
    res = {"gpu": gpu_info(), "devices": devices, "curve": "bls12_377", "h": n_h, "l": n_l, "compressed": True,
           "timing": "host clock around calls on host buffers; best of --reps after one warm-up", "runs": {}}
    print("gpu:", res["gpu"], "devices:", devices, flush=True)

    work = [bytearray(hb), bytearray(lb), bytearray(d1b), bytearray(d2b)]

    def contribute():
        S.phase2_contribute(cid, delta, work[0], work[1], True, S.CHECK_NO, work[2], work[3])

    def verify():
        S.phase2_verification(cid, hb, ha, lb, la, True, d1a, d2b, d2a, seed=seed)

    def contribute_primitives():
        for q in (hb, lb):
            u = bytearray(S.transcode(cid, S.G1, q, True, S.CHECK_NO, False))
            S.batch_mul(cid, S.G1, u, inv)
            S.transcode(cid, S.G1, bytes(u), False, S.CHECK_NO, True)
        for gid, e in ((S.G1, d1b), (S.G2, d2b)):
            u = bytearray(S.transcode(cid, gid, e, True, S.CHECK_NO, False))
            S.batch_mul(cid, gid, u, delta)
            S.transcode(cid, gid, bytes(u), False, S.CHECK_NO, True)

    g2_pair = S.transcode(cid, S.G2, d2a + d2b, True, S.CHECK_NO, False)

    def verify_primitives():
        S.check_subgroup(cid, S.G1, ha, True)
        S.check_subgroup(cid, S.G1, la, True)
        for before, after in ((hb, ha), (lb, la)):
            s, sx = S.merge_pairs(cid, S.G1, before, after, True, seed=seed, check=S.CHECK_NO)
            S.check_same_ratio(cid, s + sx, g2_pair)

    for name, fn in (("contribute_whole", contribute), ("verify_whole", verify),
                     ("contribute_primitives", contribute_primitives), ("verify_primitives", verify_primitives)):
        res["runs"][name] = timed(fn, a.reps)
        print(name, json.dumps(res["runs"][name]), flush=True)
    if devices > 1:
        ffi.init(list(range(devices)))
        for name, fn in (("contribute_sharded", contribute), ("verify_sharded", verify)):
            res["runs"][name] = timed(fn, a.reps)
            print(name, json.dumps(res["runs"][name]), flush=True)
        ffi.init([0])
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
