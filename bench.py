#!/usr/bin/env python3
"""bench.py — ONE 2^22-power BLS12-377 phase-1 ceremony round, contribute + verify, powers/s (BASELINE.json metric).

One "step" = Phase1::computation (phase1/src/computation.rs:16-193, Groth16, full mode: 2^23-1 tau_g1 +
2^22 tau_g2 / alpha_g1 / beta_g1 + beta_g2, uncompressed challenge 2 415 919 264 B -> compressed response
1 207 959 664 B) FOLLOWED BY the per-vector loop of Phase1::verification over that response
(phase1/src/verification.rs:217-411: OnlyNonZero decode, subgroup test of every element, power_pairs (s, sx) per
vector, uncompressed new challenge) and its four check_same_ratio verdicts (helpers.rs:406-424) — BASELINE.json
configs[3], the configuration the metric is quoted on.

  N ranks (torchrun, one process per GPU) SHARD THAT ONE CEREMONY by index range (SURVEY.md §8e, chunk ranges of
  phase1/src/objects/parameters.rs:248-294): rank r owns part r of N of every vector (sharding.shard_range); a verify
  shard reads one overlap element (helpers.rs:388-390); no data-path collective — the N partial (s, sx) blobs
  (960 B each) are all-gathered, rank 0 adds them (ss_phase1_reduce_partial_pairs) and runs the four pairing
  checks.  "scaling": "strong".  N = 1 is the whole ceremony on one GPU.
  value : 2^22 / (contribute_s + verify_s) with challenge and response resident in HBM, timed with CUDA events on
          the launching stream, max over ranks.
  e2e   : the same through the host-buffer C-ABI calls (ss_phase1_computation_shard +
          ss_phase1_verification_vectors_shard), pinned host buffers, every H2D / D2H copy inside the timed region;
          `e2e.pageable` repeats it with pageable host memory (what the CLI's mmaps are).
  roofline : integer-multiply pipe: executed MAC32 of the dominant kernel / its measured duration / measured peak.
  cpu_baseline : the C++ port of the reference algorithm (oracle/oracle.cpp) on the box's host cores, contribute +
          verify on a bounded sample, rank 0 at N = 1 only.

  --dump-outputs DIR : after the timed steps, rank 0 writes what the last step returned to its caller as float32 /
          float64 .npy files (see dump_outputs), so two builds can be compared output for output.  The inputs depend
          only on the arguments, and the sample of elements is fixed by DUMP_SEED.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

BLS_R = 0x12ab655e9a2ca55660b44d1e5c37b00159aa76fed00000010a11800000000001
# SURVEY.md §8(d) / BASELINE.md §3: reference-algorithm work, MAC32 per unit
W_REF_G1_MUL = 948750
W_REF_G2_MUL = 2314950
W_REF_POWER = 6109950
# Work the kernels actually EXECUTE (GLV/GLS + signed windows, glv.cuh): field multiplications / squarings per
# scalar multiplication counted on the host-emulated device code (tests/test_device_algos_emul.py::
# test_executed_work_per_scalar_mul pins them), in MAC32 = 2n^2+n per multiplication, (3n^2+3n)/2 per squaring (n = 12).
W_EXEC_G1_MUL = 775 * 300 + 890 * 234
W_EXEC_G2_MUL = 3200 * 300
METRIC = "phase1 contribute+verify G1+G2 powers/sec at 2^22 (1/2/4/8 B200), bit-exact"
VECTORS = ("tau_g1", "tau_g2", "alpha_g1", "beta_g1", "beta_g2")
DUMP_SEED = 20261020
DUMP_ELEMENTS = 8192  # per vector: 8192 x 720 B of response + new challenge = 24 MB as float32


def derive_scalar(seed: bytes, label: bytes) -> int:
    return int.from_bytes(hashlib.blake2b(seed + b"/" + label, digest_size=64).digest(), "little") % (BLS_R - 1) + 1


def keys(seed: bytes):
    return tuple(derive_scalar(seed, l) for l in (b"tau", b"alpha", b"beta"))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU, sampled every 200 ms while running."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        pw = [float(r[2]) for r in self.rows if len(r) >= 7 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def workload_text(k, acc_len, resp_len):
    return (f"ONE phase1 round over 2^{k} powers, BLS12-377 Groth16 full mode: contribute (Phase1::computation, uncompressed "
            f"challenge {acc_len} B -> compressed response {resp_len} B) + verify (per-vector loop of Phase1::verification: "
            f"OnlyNonZero decode, subgroup test, power_pairs, uncompressed new challenge {acc_len} B, four check_same_ratio)")


def cpu_round(O, R, k, k0, k1, decode_passes=2):
    """One contribute + verify round of a 2^k-power ceremony on the CPU port.  Returns (contribute_s, verify_s)."""
    p = R.Phase1Parameters(R.BLS12_377, k, 256)
    acc = bytes(R.phase1_initialization(p, False))
    acc = O.phase1_computation(0, acc, p.get_length(False), False, False, 3, p.g1_chunk_size, p.other_chunk_size, 0, *k0)
    t = time.perf_counter()
    resp = O.phase1_computation(0, acc, p.get_length(True), False, True, 3, p.g1_chunk_size, p.other_chunk_size, 0, *k1)
    tc = time.perf_counter() - t
    t = time.perf_counter()
    O.phase1_verification_vectors(0, resp, True, p.get_length(False), False, p.g1_chunk_size, p.other_chunk_size,
                                  decode_passes=decode_passes)
    tv = time.perf_counter() - t
    return tc, tv


def cpu_sample_text(k, tc, tv):
    return (f"one 2^{k}-power BLS12-377 round: Phase1::computation {tc:.2f} s + verification loop {tv:.2f} s (reference "
            f"algorithm: double-and-add batch_exp, Tonelli-Shanks decode run twice per element as accumulator.rs:102-106 + "
            f":64-68 do, r*P subgroup test, two signed-bucket msm_bigint over full-width random scalars); work is linear in "
            f"the number of powers")


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm (C++ port; the Rust reference cannot be built in this image) on
    all host cores, one bounded sample of the workload (a whole small ceremony round) per step."""
    if rank != 0:
        return
    import coracle as O
    import pyref as R
    O.set_threads(len(os.sched_getaffinity(0)))  # torchrun exports OMP_NUM_THREADS=1: use every host core anyway
    cores = O.threads()
    k = args.ref_power
    k0, k1 = keys(b"bench-0"), keys(b"bench-1")
    times = []
    for it in range(args.warmup + args.steps):
        tc, tv = cpu_round(O, R, k, k0, k1)
        if it >= args.warmup:
            times.append((tc, tv))
    total = sum(a + b for a, b in times)
    v = (1 << k) * len(times) / total
    tcm, tvm = sum(a for a, _ in times) / len(times), sum(b for _, b in times) / len(times)
    K = args.power
    prm = R.Phase1Parameters(R.BLS12_377, K, 256)
    restore_stdout()
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "powers/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": total / len(times) * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_text(K, prm.get_length(False), prm.get_length(True)) +
                               " — reference algorithm on host cores, bounded sample", "sample_power": k},
        "cpu_baseline": {"value": v, "unit": "powers/s", "cores": cores, "kind": "port", "sample": cpu_sample_text(k, tcm, tvm),
                         "fq_mul_ns": round(O.fq_mul_ns(), 1), "asm_mul": O.has_asm_mul(),
                         "contribute_powers_per_s": (1 << k) / tcm, "verify_powers_per_s": (1 << k) / tvm},
        "e2e": {"value": v, "unit": "powers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def cpu_baseline(budget_s=20.0):
    import coracle as O
    import pyref as R
    O.set_threads(len(os.sched_getaffinity(0)))
    cores = O.threads()
    k0, k1 = keys(b"bench-0"), keys(b"bench-1")
    cpu_round(O, R, 6, k0, k1)  # thread pool / page warm-up
    tc, tv = cpu_round(O, R, 10, k0, k1)
    k = 10
    while k < 16 and (tc + tv) * (1 << (k + 1 - 10)) <= budget_s:
        k += 1
    if k > 10:
        tc, tv = cpu_round(O, R, k, k0, k1)
    return {"value": (1 << k) / (tc + tv), "unit": "powers/s", "cores": cores, "kind": "port",
            "sample": cpu_sample_text(k, tc, tv), "fq_mul_ns": round(O.fq_mul_ns(), 1), "asm_mul": O.has_asm_mul(),
            "contribute_powers_per_s": (1 << k) / tc, "verify_powers_per_s": (1 << k) / tv}


NCU_FULL = os.path.join("profiles", "r02_ncu_full_final.json")


def ncu_traffic(name, d):
    """`traffic` of the dominant kernel from the committed same-round `ncu --set full` capture (dram__bytes_read.sum +
    dram__bytes_write.sum of its largest launch there), scaled by elements to this run's average launch — or null."""
    none = {"traffic": None, "traffic_note": "no ncu --set full capture of this kernel under %s" % NCU_FULL}
    try:
        cap = json.load(open(os.path.join(ROOT, NCU_FULL)))
        tag = "k_scalar_mul<Bls377G2>" if ".g2" in name else "k_scalar_mul<Bls377G1>"
        best = None
        for rec in cap["launches"]:
            if tag in rec["Kernel Name"]:
                grid = int(rec["Grid Size"].strip("()").split(",")[0])
                block = int(rec["Block Size"].strip("()").split(",")[0])
                if best is None or grid > best[0]:
                    to_b = lambda t: float(t.split()[0]) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[t.split()[1]]  # noqa: E731
                    best = (grid, grid * block, to_b(rec["dram__bytes_read.sum"]) + to_b(rec["dram__bytes_write.sum"]))
        if not best or best[1] < 1024:
            return none
        per_launch = d["elements"] / max(1, d["launches"])
        return {"traffic": best[2] / best[1] * per_launch, "traffic_unit": "bytes per launch",
                "traffic_source": "%s: %.0f MB DRAM read+write for a %d-thread launch of this kernel (ncu --set full, same build), "
                                  "scaled by elements to this run's %.0f-element launches; algorithmic bytes are %d per element — "
                                  "the excess is the per-thread window table and Jacobian spills in local memory of an "
                                  "integer-pipe-bound kernel" % (NCU_FULL, best[2] / 1e6, best[1], per_launch,
                                                                  (192 + 96) if ".g2" in name else (96 + 48))}
    except Exception as exc:
        none["traffic_note"] += " (%r)" % (exc,)
        return none


def run_extras(S, R, O, bw6_power, phase2_log2):
    """One-step measurements of the other BASELINE configs through the host-buffer C ABI, reported beside the headline
    (`extras`), never part of `value`:  C3 = BW6-761 phase-1 verify (subgroup checks + power_pairs MSM + the four device
    pairing verdicts) of a 2^bw6_power-power response, C5 = phase 2's delta^-1 batch_mul of a 2^phase2_log2-element
    query + its merge_pairs ratio MSM.  Each leg: one warm-up pass, one timed pass, a parity spot check."""
    out = {}
    cv, cid = R.BW6_761, S.BW6_761
    k = bw6_power
    N = 1 << k
    rp, sp = R.Phase1Parameters(cv, k, 256), S.Phase1Parameters(cid, k, 256)
    sc = lambda lab: int.from_bytes(hashlib.blake2b(lab, digest_size=64).digest(), "little") % (cv.r - 2) + 2  # noqa: E731
    k0, k1 = [sc(b"bw6-0-%d" % i) for i in range(3)], [sc(b"bw6-1-%d" % i) for i in range(3)]
    blank = S.phase1_initialization(sp, False)
    chal = bytearray(sp.get_length(False))
    S.phase1_computation(sp, blank, chal, False, False, S.CHECK_NO, *k0)
    del blank
    resp = bytearray(sp.get_length(True))
    S.phase1_computation(sp, chal, resp, False, True, S.CHECK_NO, *k1)  # warm-up of the contribute leg
    t = time.perf_counter()
    S.phase1_computation(sp, chal, resp, False, True, S.CHECK_NO, *k1)
    t_c = time.perf_counter() - t
    o, _, sz = rp.split_offsets(False)[0]
    oo, _, szo = rp.split_offsets(True)[0]
    i0 = 1234 % (2 * N - 5)
    ok = bytes(resp[oo + i0 * szo:oo + (i0 + 4) * szo]) == O.apply_powers(1, 0, bytes(chal[o + i0 * sz:o + (i0 + 4) * sz]), False, 3,
                                                                         True, 4, tau=k1[0], first_power=i0)
    del chal
    progress("extras: C3 contribute done")
    newc = bytearray(sp.get_length(False))
    seed = bytes(range(32))
    S.phase1_verification_ratios(sp, resp, True, newc, False, seed=seed)
    t = time.perf_counter()
    S.phase1_verification_ratios(sp, resp, True, newc, False, seed=seed)  # raises on a bad verdict
    t_v = time.perf_counter() - t
    ok = ok and bytes(newc[o + i0 * sz:o + (i0 + 4) * sz]) == O.transcode(1, 0, bytes(resp[oo + i0 * szo:oo + (i0 + 4) * szo]), True, 3, False, 4)
    progress("extras: C3 measured")
    out["C3_bw6_761_phase1"] = {"power": k, "verify_powers_per_s": N / t_v, "verify_ms": t_v * 1e3, "contribute_powers_per_s": N / t_c,
                                "contribute_ms": t_c * 1e3, "verdict": True, "parity_spot_check": bool(ok),
                                "what": "host buffers; verify = ss_phase1_verification_ratios (vectors + 4 device pairing checks)"}
    del newc, resp
    # C5
    cv, cid, g = R.BLS12_377, S.BLS12_377, R.BLS12_377.g1
    n = 1 << phase2_log2
    sc = lambda lab: int.from_bytes(hashlib.blake2b(lab, digest_size=64).digest(), "little") % (cv.r - 2) + 2  # noqa: E731
    h_before = S.apply_powers(cid, S.G1, g.encode(g.gen, False) * n, False, S.CHECK_NO, False, n, tau=sc(b"p2-tau"), first_power=1)
    dinv = sc(b"p2-delta-inv")
    buf = bytearray(h_before)
    S.batch_mul(cid, S.G1, buf, dinv)
    buf[:] = h_before
    t = time.perf_counter()
    S.batch_mul(cid, S.G1, buf, dinv)
    t_mul = time.perf_counter() - t
    ok = bytes(buf[:96 * 8]) == O.apply_powers(0, 0, h_before[:96 * 8], False, 3, False, 8, powers=[dinv] * 8)
    after = bytes(buf)
    S.merge_pairs(cid, S.G1, h_before, after, False, seed=bytes(range(32)))
    t = time.perf_counter()
    s_, sx_ = S.merge_pairs(cid, S.G1, h_before, after, False, seed=bytes(range(32)))
    t_mp = time.perf_counter() - t
    rok = O.apply_powers(0, 0, s_, False, 3, False, 1, powers=[dinv]) == sx_
    out["C5_phase2_query"] = {"n": n, "batch_mul_elements_per_s": n / t_mul, "batch_mul_ms": t_mul * 1e3,
                              "merge_pairs_pairs_per_s": n / t_mp, "merge_pairs_ms": t_mp * 1e3, "parity_spot_check": bool(ok),
                              "ratio_check": bool(rok), "what": "host buffers; ss_batch_mul / ss_merge_pairs on uncompressed G1"}
    return out


def dump_sample(count, vector):
    """Sorted element indices of `vector` that --dump-outputs writes: all of them up to DUMP_ELEMENTS, else a fixed
    seeded sample."""
    import numpy as np
    if count <= DUMP_ELEMENTS:
        return np.arange(count)
    return np.sort(np.random.default_rng([DUMP_SEED, vector]).choice(count, DUMP_ELEMENTS, replace=False))


def dump_outputs(out_dir, buffers, pairs, accepted, rank, world, dist=None):
    """Writes what one round returns to its caller:
      <buffer>_<vector>.npy  float32 [elements, element bytes]: the bytes of the dump_sample elements of each vector of
                             every (buffer name, device uint8 tensor, sharding.vector_offsets) in `buffers`;
      ratio_pairs.npy        float32 bytes of the (s, sx) blob the four ratio checks read (reduced over ranks);
      verdict.npy            float64 [1]: 1 when the four checks accepted the response.
    Each rank contributes the sampled elements of its own shard, so the files do not depend on the number of GPUs."""
    import numpy as np
    import torch
    from snark_setup_b200 import sharding
    arrays = {}
    for v, name in enumerate(VECTORS):
        for label, buf, offs in buffers:
            o, cnt, sz = offs[v]
            idx = torch.from_numpy(dump_sample(cnt, v)).to(buf.device)
            rows = buf[o:o + cnt * sz].view(cnt, sz).index_select(0, idx).float()
            s, e = sharding.shard_range(cnt, rank, world)
            rows[(idx < s) | (idx >= e)] = 0  # computed by another rank
            if world > 1:
                dist.all_reduce(rows)
            arrays[f"{label}_{name}"] = rows.cpu().numpy()
    if rank != 0:
        return
    arrays["ratio_pairs"] = np.frombuffer(pairs, dtype=np.uint8).astype(np.float32)
    arrays["verdict"] = np.array([1.0 if accepted else 0.0])
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


_STDOUT_FD = None
_T0 = time.perf_counter()


def progress(msg):
    """leg boundaries on stderr (stdout carries the one JSON line only)"""
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench %7.1fs] %s" % (time.perf_counter() - _T0, msg), file=sys.stderr, flush=True)


def restore_stdout():
    global _STDOUT_FD
    if _STDOUT_FD is not None:
        sys.stdout.flush()
        os.dup2(_STDOUT_FD, 1)
        os.close(_STDOUT_FD)
        _STDOUT_FD = None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--power", type=int, default=22, help="log2 powers of the ceremony (default 22 = the metric's configuration)")
    ap.add_argument("--ref-power", type=int, default=12, help="log2 powers of one reference-arm step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the one-step C3 (BW6-761) / C5 (phase 2) measurements")
    ap.add_argument("--extras-bw6-power", type=int, default=21)
    ap.add_argument("--extras-phase2-log2", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's response, new challenge, ratio pairs and verdict to DIR/*.npy")
    ap.add_argument("--cpu-baseline-only", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.cpu_baseline_only:
        print(json.dumps(cpu_baseline()), flush=True)
        return
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries the ONE JSON line and nothing else: anything native libraries write to fd 1 while the
    # bench runs (NCCL prints its version line there when NCCL_DEBUG=VERSION) is sent to stderr instead.
    global _STDOUT_FD
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch
    import torch.distributed as dist
    import snark_setup_b200 as S
    from snark_setup_b200 import ffi, sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the CUDA path is the product, there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    ffi.init([local_rank])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return sharding.max_over_ranks(x, dist if world > 1 else None, dev)

    def all_ok(flag):
        if world == 1:
            return bool(flag)
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item())

    k = args.power
    N = 1 << k
    cid = S.BLS12_377
    prm = S.Phase1Parameters(cid, k, 256)
    acc_len, resp_len = prm.get_length(False), prm.get_length(True)
    shard = (rank, world)
    seed = hashlib.blake2b(b"bench-rho", digest_size=32).digest()

    # ---- synthetic ceremony state (every rank builds the whole of it, untimed): generators -> contribution
    #      "bench-0" = the challenge; one whole contribution "bench-1" = the response the verify shards read --------
    import pyref as R
    g1, g2 = R.BLS12_377.g1, R.BLS12_377.g2
    g1b = torch.frombuffer(bytearray(g1.encode(g1.gen, False)), dtype=torch.uint8).to(dev)
    g2b = torch.frombuffer(bytearray(g2.encode(g2.gen, False)), dtype=torch.uint8).to(dev)
    blank = torch.cat([torch.zeros(64, dtype=torch.uint8, device=dev), g1b.repeat(2 * N - 1), g2b.repeat(N),
                       g1b.repeat(N), g1b.repeat(N), g2b])
    assert blank.numel() == acc_len
    challenge = torch.empty(acc_len, dtype=torch.uint8, device=dev)
    response = torch.zeros(resp_len, dtype=torch.uint8, device=dev)
    newc = torch.zeros(acc_len, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    k0, k1 = keys(b"bench-0"), keys(b"bench-1")
    S.phase1_computation_dev(prm, blank.data_ptr(), acc_len, challenge.data_ptr(), acc_len, False, False, S.CHECK_NO,
                             *k0, stream=stream)
    del blank
    torch.cuda.empty_cache()
    S.phase1_computation_dev(prm, challenge.data_ptr(), acc_len, response.data_ptr(), resp_len, False, True, S.CHECK_NO,
                             *k1, stream=stream)
    torch.cuda.synchronize()
    # g1_check / g2_check = first two tau_g1 / tau_g2 elements of the response (verification.rs:58-71), read once
    offs_c = sharding.vector_offsets(2 * N - 1, N, True)
    offs_u = sharding.vector_offsets(2 * N - 1, N, False)
    g1_check = S.transcode(cid, S.G1, response[offs_c[0][0]:offs_c[0][0] + 96].cpu().numpy().tobytes(), True, S.CHECK_FULL, False, 2)
    g2_check = S.transcode(cid, S.G2, response[offs_c[1][0]:offs_c[1][0] + 192].cpu().numpy().tobytes(), True, S.CHECK_FULL, False, 2)
    nblob = S.pairs_size(cid)
    d_blob = torch.zeros(nblob, dtype=torch.uint8, device=dev)
    d_all = torch.zeros(nblob * world, dtype=torch.uint8, device=dev)
    last_pairs = [None]  # rank 0: the whole (s, sx) blob of the latest verification

    def verdict(blob):
        """partial blob of this rank -> (gather) -> rank 0: sum + the four check_same_ratio.  Returns True / False / None."""
        if world > 1:
            d_blob.copy_(torch.frombuffer(bytearray(blob), dtype=torch.uint8))
            dist.all_gather_into_tensor(d_all, d_blob)
            if rank != 0:
                return None
            blob = S.phase1_reduce_partial_pairs(cid, [d_all[i * nblob:(i + 1) * nblob].cpu().numpy().tobytes()
                                                       for i in range(world)], raw=True)
        last_pairs[0] = blob
        try:
            S.phase1_check_ratio_pairs(cid, blob, g1_check, g2_check)
            return True
        except S.InvalidRatio:
            return False

    def contribute_dev():
        S.phase1_computation_dev(prm, challenge.data_ptr(), acc_len, response.data_ptr(), resp_len, False, True,
                                 S.CHECK_NO, *k1, stream=stream, shard=shard)

    def verify_dev():
        blob = S.phase1_verification_vectors_dev(prm, response.data_ptr(), resp_len, True, newc.data_ptr(), acc_len,
                                                 False, seed=seed, stream=stream, shard=shard, raw=True)
        return verdict(blob)

    for _ in range(args.warmup):
        contribute_dev()
        verify_dev()
    # ---- timed region: device-resident ---------------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    ffi.profile_reset()
    barrier()
    sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps + 1)]
    verdicts = []
    ev[0].record()
    for i in range(args.steps):
        contribute_dev()
        ev[2 * i + 1].record()
        verdicts.append(verify_dev())
        ev[2 * i + 2].record()
    barrier()
    dev_ms = max_over_ranks(ev[0].elapsed_time(ev[-1]))
    c_ms = max_over_ranks(sum(ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.steps)))
    v_ms = max_over_ranks(sum(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(args.steps)))
    clocks = sampler.stop()
    launches = ffi.profile_launches()
    value = N * args.steps / (dev_ms * 1e-3)
    verdict_ok = all(v is True for v in verdicts) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [("response", response, offs_c), ("new_challenge", newc, offs_u)], last_pairs[0],
                     verdicts[-1], rank, world, dist)
        progress("outputs of the last timed step written to %s" % args.dump_outputs)

    # per-kernel durations for the roofline: one extra round with the vectors SERIALISED on one stream, so the
    # event brackets around each launch measure that kernel alone (in the timed region above the five vectors
    # run on concurrent streams and their kernels time-slice the SMs)
    def profiled(fn):
        ffi.set_concurrent_vectors(False)
        fn()
        ffi.profile_reset()
        ffi.profile_enable(True)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ffi.profile_enable(False)
        pr = ffi.profile_read()
        ffi.set_concurrent_vectors(True)
        return pr, a.elapsed_time(b)

    prof_c, serial_c_ms = profiled(contribute_dev)
    prof_v, serial_v_ms = profiled(verify_dev)

    # ---- parity spot checks against the oracle (test infrastructure used as the checker only): a slice of EVERY
    #      vector inside this rank's shard — response bytes vs the CPU port, new challenge vs the transcoded response
    import coracle as O
    cnts = (2 * N - 1, N, N, N)
    grp = (0, 1, 0, 0)
    coeffs = (None, None, k1[1], k1[2])
    n_chk = 8
    ok = True
    for v in range(4):
        s, e = sharding.shard_range(cnts[v], rank, world)
        idx = s + (123457 * (v + 1)) % max(1, e - s - n_chk)
        (oc, _, szc), (ou, _, szu) = offs_c[v], offs_u[v]
        cin = challenge[ou + idx * szu: ou + (idx + n_chk) * szu].cpu().numpy().tobytes()
        got = response[oc + idx * szc: oc + (idx + n_chk) * szc].cpu().numpy().tobytes()
        want = O.apply_powers(0, grp[v], cin, False, 3, True, n_chk, tau=k1[0], first_power=idx, coeff=coeffs[v])
        ok = ok and got == want
        got_nc = newc[ou + idx * szu: ou + (idx + n_chk) * szu].cpu().numpy().tobytes()
        ok = ok and got_nc == O.transcode(0, grp[v], got, True, 3, False, n_chk)
    if rank == 0:  # beta_g2 belongs to shard 0
        (oc, _, szc), (ou, _, szu) = offs_c[4], offs_u[4]
        cin = challenge[ou: ou + szu].cpu().numpy().tobytes()
        got = response[oc: oc + szc].cpu().numpy().tobytes()
        ok = ok and got == O.apply_powers(0, 1, cin, False, 3, True, 1, powers=[k1[2]])
        ok = ok and newc[ou: ou + szu].cpu().numpy().tobytes() == O.transcode(0, 1, got, True, 3, False, 1)
    parity = all_ok(ok)

    progress("device-resident legs and parity spot check done")
    # ---- e2e: host buffers through the C ABI, every copy inside the timed region ---------------------------------
    e2e = None
    if not args.no_e2e:
        sh_in = sum(sharding.shard_bytes(cnts[v], rank, world, offs_u[v][2]) for v in range(4)) + (192 if rank == 0 else 0)
        sh_out = sum(sharding.shard_bytes(cnts[v], rank, world, offs_c[v][2]) for v in range(4)) + (96 if rank == 0 else 0)
        overlap = sum(offs_c[v][2] for v in range(4) if sharding.shard_range(cnts[v], rank, world)[1] < cnts[v])

        def run_e2e(pinned, steps):
            h_chal = torch.empty(acc_len, dtype=torch.uint8, pin_memory=pinned)
            h_resp = torch.empty(resp_len, dtype=torch.uint8, pin_memory=pinned)
            h_newc = torch.empty(acc_len, dtype=torch.uint8, pin_memory=pinned)
            h_chal.copy_(challenge)
            h_resp.copy_(response)  # the overlap elements of the neighbouring shard are part of the input
            torch.cuda.synchronize()
            a_chal, a_resp, a_newc = h_chal.numpy(), h_resp.numpy(), h_newc.numpy()

            def round_():
                S.phase1_computation(prm, a_chal, a_resp, False, True, S.CHECK_NO, *k1, shard=shard)
                blob = S.phase1_verification_vectors(prm, a_resp, True, a_newc, False, seed=seed, shard=shard, raw=True)
                return verdict(blob)

            for _ in range(2):  # warm-up: staging slabs of the host path are (re)grown here, not in the timed region
                round_()
            barrier()
            t0 = time.perf_counter()
            vd = [round_() for _ in range(steps)]
            barrier()
            dt = max_over_ranks(time.perf_counter() - t0)
            # the host path must produce the bytes of the device path
            s, e = sharding.shard_range(cnts[0], rank, world)
            oc, _, szc = offs_c[0]
            same = bool(torch.equal(h_resp[oc + s * szc: oc + e * szc], response[oc + s * szc: oc + e * szc].cpu()))
            ou, _, szu = offs_u[0]
            same = same and bool(torch.equal(h_newc[ou + s * szu: ou + e * szu], newc[ou + s * szu: ou + e * szu].cpu()))
            return dt, all_ok(same), (all(v is True for v in vd) if rank == 0 else None)

        e2e_steps = max(1, min(args.steps, 5))
        dt, same, vd = run_e2e(True, e2e_steps)
        e2e = {"value": N * e2e_steps / dt, "unit": "powers/s",
               "h2d_bytes_per_step": int(sh_in + sh_out + overlap), "d2h_bytes_per_step": int(sh_out + sh_in),
               "bytes_are": "this rank's shard: contribute challenge H2D + response D2H, verify response H2D (+ overlap elements) "
                            "+ new challenge D2H; whole ceremony = N x",
               "steps": e2e_steps, "ms_per_step": dt / e2e_steps * 1e3, "host_memory": "pinned",
               "matches_device_path": same, "verdict": vd}
        progress("e2e (pinned) done")
        if not args.no_pageable:
            p_steps = max(1, min(args.steps, 3))
            dt, same, vd = run_e2e(False, p_steps)
            e2e["pageable"] = {"value": N * p_steps / dt, "unit": "powers/s", "steps": p_steps,
                               "ms_per_step": dt / p_steps * 1e3, "matches_device_path": same, "verdict": vd}

    progress("e2e legs done")
    # ---- roofline of the dominant kernels ------------------------------------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    imad = None
    try:
        imad = json.load(open(os.path.join(ROOT, "profiles", "imad_peak.json")))
    except Exception:
        pass
    mac_peak = (imad or {}).get("mac32_tps", 9.2)  # T MAC32/s: 18.4 T IMAD/s / 2 IMAD per MAC32
    peak_src = ("measured IMAD microbenchmark on this pool (profiles/imad_peak.json: 18.4 T IMAD/s / 2 IMAD per MAC32)"
                if imad else "fallback 18.4 T IMAD/s / 2")

    def executed(name, d):
        w = W_EXEC_G2_MUL if ".g2" in name else W_EXEC_G1_MUL
        ach = w * d["elements"] / (d["ms"] * 1e-3) * 1e-12
        return {"kernel": name, "mac32_per_element": w, "elements": d["elements"], "launches": d["launches"],
                "avg_launch_ms": d["ms"] / max(1, d["launches"]), "achieved": ach, "frac": ach / mac_peak}

    roofline = None
    smul = {kk: vv for kk, vv in prof_c.items() if kk.startswith("k_scalar_mul")}
    if smul:
        name, d = max(smul.items(), key=lambda kv: kv[1]["ms"])
        total_ms = sum(v["ms"] for v in prof_c.values())
        ex = executed(name, d)
        w_ref = W_REF_G2_MUL if ".g2" in name else W_REF_G1_MUL
        roofline = {
            "bound": "int32-imad", "kernel": name, "unit": "TMAC32/s", "peak": mac_peak, "peak_source": peak_src,
            "what": "EXECUTED multiply-accumulates (GLV/GLS algorithm, counted on the emulated device code, pinned by "
                    "tests/test_device_algos_emul.py) of the dominant kernel / its measured duration / measured peak",
            "achieved": ex["achieved"], "frac": ex["frac"], "mac32_per_element": ex["mac32_per_element"],
            "avg_launch_ms": ex["avg_launch_ms"], "kernel_share_of_contribute_step": d["ms"] / total_ms,
            **ncu_traffic(name, d),
            "second_kernel": next((executed(n2, d2) for n2, d2 in smul.items() if n2 != name), None),
            "vs_reference_algorithm": {
                "what": "W_ref (reference double-and-add, SURVEY §8d) x elements / duration / peak — a speed-up-vs-reference-"
                        "algorithm figure, may exceed 1 because GLV does ~2.15x less work; NOT a utilisation",
                "kernel_frac": w_ref * d["elements"] / (d["ms"] * 1e-3) * 1e-12 / mac_peak,
                "contribute_step_frac": W_REF_POWER * (N * args.steps / (c_ms * 1e-3)) * 1e-12 / mac_peak / world},
            "hbm": {"algorithmic_GBps_per_gpu": 2 * (acc_len + resp_len) / world * args.steps / (dev_ms * 1e-3) * 1e-9,
                    "peak_GBps": peaks.get("hbm_gbs")},
            "serialised_ms": {"contribute": serial_c_ms, "verify": serial_v_ms},
            "kernels_ms_contribute": {kk: round(vv["ms"], 3) for kk, vv in sorted(prof_c.items())},
            "kernels_ms_verify": {kk: round(vv["ms"], 3) for kk, vv in sorted(prof_v.items())}}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # in a child process: the CPU port is test infrastructure, and nothing it does (or a crash in it) may cost the
        # headline line
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only"], capture_output=True, text=True,
                               timeout=600)
            lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
            cpu = json.loads(lines[-1]) if r.returncode == 0 and lines else {"error": "exit %d: %s" % (r.returncode, r.stderr[-200:])}
        except Exception as exc:
            cpu = {"error": repr(exc)[:300]}
        progress("cpu baseline done")

    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        del challenge, response, newc
        torch.cuda.empty_cache()
        try:
            extras = run_extras(S, R, O, args.extras_bw6_power, args.extras_phase2_log2)
        except Exception as exc:  # the headline line must not depend on the side measurements
            extras = {"error": repr(exc)[:300]}
        progress("extras done")

    if rank == 0:
        restore_stdout()
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": "powers/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_text(k, acc_len, resp_len),
                       "sharding": f"index-range shard {world} ways of the one ceremony (rank r = part r of every vector, one "
                                   f"overlap element per verify shard); partial (s, sx) all-gathered ({nblob} B per rank) and "
                                   f"summed on rank 0; no data-path collective",
                       "cache": "per-rank inputs (>= %d MB) larger than L2 (126 MB); no flush needed" % ((acc_len + resp_len) // world >> 20),
                       "synthetic_input": "generators -> contribution keyed 'bench-0' (challenge) -> timed contribution 'bench-1' "
                                          "-> timed verification of that response"},
            "legs": {"contribute": {"powers_per_s": N * args.steps / (c_ms * 1e-3), "ms_per_step": c_ms / args.steps},
                     "verify": {"powers_per_s": N * args.steps / (v_ms * 1e-3), "ms_per_step": v_ms / args.steps,
                                "includes": "partial-sum all-gather, reduction and the four device pairing checks on rank 0"}},
            "clocks": clocks, "gpu_launches": int(launches), "verdict_all_steps": verdict_ok,
            "e2e": e2e, "roofline": roofline, "cpu_baseline": cpu, "parity_spot_check": parity, "extras": extras,
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
