#!/usr/bin/env python3
"""Times Groth16Params::new (ss_groth16_params_new: four group IFFTs + the H query) on MNT4-753 and MNT6-753.

For each size 2^k the accumulator is a real one: pyref's blank (G2 slots hold its derived generator) contributed to
once on the device with random keys, so the transforms see unstructured points.  Each size is warmed up once and then
timed over --reps calls (host clock around the call, which returns after a device synchronise).  Sizes are tried in
increasing order per curve and the curve stops once a call exceeds --max-call-s.  MNT6-753 has no radix-2 domain above
2^15.

    python tools/mnt_phase2_bench.py --out results.json
"""
import argparse
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

CURVES = {"mnt4_753": S.MNT4_753, "mnt6_753": S.MNT6_753}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return "unknown (%s)" % e


def accumulator(curve, power, rng):
    cv = R.curve_by_name(curve)
    rp = R.Phase1Parameters(cv, power, 1 << 14)
    sp = S.Phase1Parameters(CURVES[curve], power, 1 << 14)
    blank = bytes(R.phase1_initialization(rp, False))
    acc = bytearray(sp.get_length(False))
    S.phase1_computation(sp, blank, acc, False, False, S.CHECK_NO, *[rng.randrange(2, cv.r) for _ in range(3)])
    return sp, bytes(acc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mnt4-powers", default="10,12,14,16")
    ap.add_argument("--mnt6-powers", default="10,12,14,15")
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--max-call-s", type=float, default=60.0, help="stop growing a curve's size after a call this long")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rng = random.Random(2024)
    res = {"gpu": gpu_info(), "timing": "host clock around ss_groth16_params_new, uncompressed in and out", "runs": []}
    print("gpu:", res["gpu"], flush=True)
    for curve, powers in (("mnt4_753", a.mnt4_powers), ("mnt6_753", a.mnt6_powers)):
        for k in [int(x) for x in powers.split(",") if x]:
            t0 = time.perf_counter()
            sp, acc = accumulator(curve, k, rng)
            t_acc = time.perf_counter() - t0
            m = 1 << k
            t0 = time.perf_counter()
            S.groth16_params_new(sp, acc, False, m, False)  # warm-up (module load, lane allocation)
            t_first = time.perf_counter() - t0
            ts = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                S.groth16_params_new(sp, acc, False, m, False)
                ts.append(time.perf_counter() - t0)
            run = {"curve": curve, "log2_domain": k, "accumulator_build_s": round(t_acc, 3), "first_call_s": round(t_first, 3),
                   "call_s": [round(t, 4) for t in ts], "best_s": round(min(ts), 4),
                   # four IFFTs of m points: ~ (log m - 2) * m / 2 + 2 twiddle multiplications each (fft.cuh)
                   "scalar_muls_per_vector": (k - 2) * m // 2 + 2 if k >= 2 else 2}
            res["runs"].append(run)
            print(json.dumps(run), flush=True)
            if min(ts) > a.max_call_s:
                break
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
