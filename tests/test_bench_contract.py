"""bench.py contract checks: the reference arm (`--impl reference`) prints exactly one JSON line on stdout with the keys
a caller reads, the b200 arm refuses to run without a CUDA device (no CPU fallback), and --dump-outputs writes a fixed
sample of what the timed round computed, whatever the number of ranks (the last test needs the GPU)."""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--ref-power", "6"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == base["metric"] and d["unit"] == "powers/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "powers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1", "--ref-power", "6"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.skipif(_have_gpu(), reason="box has a GPU")
def test_b200_arm_needs_a_gpu():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_roofline_traffic_comes_from_the_named_capture():
    """`roofline.traffic` is read from the committed same-round ncu --set full summary and names it; a kernel without
    a capture gives null, never a made-up figure."""
    b = _load_bench()
    t = b.ncu_traffic("k_scalar_mul<bls12_377.g1>", {"elements": 1 << 24, "launches": 16, "ms": 1000.0})
    cap = json.load(open(os.path.join(ROOT, b.NCU_FULL)))
    rec = max((r for r in cap["launches"] if "k_scalar_mul<Bls377G1>" in r["Kernel Name"]),
              key=lambda r: int(r["Grid Size"].strip("()").split(",")[0]))
    threads = int(rec["Grid Size"].strip("()").split(",")[0]) * int(rec["Block Size"].strip("()").split(",")[0])
    mb = float(rec["dram__bytes_read.sum"].split()[0]) + float(rec["dram__bytes_write.sum"].split()[0])
    assert rec["dram__bytes_read.sum"].split()[1] == "Mbyte" and rec["dram__bytes_write.sum"].split()[1] == "Mbyte"
    assert abs(t["traffic"] - mb * 1e6 / threads * (1 << 20)) < 1e-3 * t["traffic"]
    assert b.NCU_FULL in t["traffic_source"]
    # only a one-thread G2 launch (beta_g2) is in the capture: null, with the reason
    none = b.ncu_traffic("k_scalar_mul<bls12_377.g2>", {"elements": 1 << 20, "launches": 2, "ms": 100.0})
    assert none["traffic"] is None and "traffic_note" in none


def test_committed_bench_lines_carry_the_contract_keys():
    """The evidence files of the final build are what bench.py printed: one JSON line with every key of the contract."""
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    for name, n in (("r02_bench_default_final.json", 1), ("r02_bench_final_n2.json", 2), ("r02_bench_final_n4.json", 4),
                    ("r02_bench_final_n8.json", 8)):
        lines = [l for l in open(os.path.join(ROOT, "profiles", name)) if l.startswith("{")]
        assert len(lines) == 1, name
        d = json.loads(lines[0])
        for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                    "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
            assert key in d, (name, key)
        assert d["metric"] == base["metric"] and d["n_gpus"] == n and d["warmup"] >= 3 and d["gpu_launches"] > 0
        assert "2^22" in d["config"]["workload"] and d["scaling"] == "strong" and d["vs_baseline"] is None
        assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"] * 1.01
        assert abs(d["value"] - (1 << 22) / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
        r = d["roofline"]
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0 < r["frac"] < 1
        assert not d["clocks"]["reasons"] and d["verdict_all_steps"] is True and d["parity_spot_check"] is True
        if n == 1:
            assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1


def _round_buffers(k):
    """(name, uint8 tensor, vector offsets) of a random compressed response and uncompressed new challenge at 2^k."""
    import torch
    from snark_setup_b200 import sharding
    n = 1 << k
    offs_c, offs_u = sharding.vector_offsets(2 * n - 1, n, True), sharding.vector_offsets(2 * n - 1, n, False)
    g = torch.Generator().manual_seed(k)
    return [(name, torch.randint(0, 256, (offs[-1][0] + offs[-1][2],), dtype=torch.uint8, generator=g), offs)
            for name, offs in (("response", offs_c), ("new_challenge", offs_u))]


def _dump_worker(rank, world, port, out):
    import torch.distributed as dist
    from snark_setup_b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    bufs = _round_buffers(13)
    for _, t, offs in bufs:  # a rank holds only its own shard of the round
        for o, cnt, sz in offs:
            s, e = sharding.shard_range(cnt, rank, world)
            t[o:o + s * sz] = 0
            t[o + e * sz:o + cnt * sz] = 0xFF
    _load_bench().dump_outputs(out, bufs, bytes(range(240)) * 4, True, rank, world, dist)
    dist.destroy_process_group()


def _load_dir(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_is_a_fixed_sample_independent_of_ranks(tmp_path):
    import torch.multiprocessing as mp
    b = _load_bench()
    bufs = _round_buffers(13)
    b.dump_outputs(str(tmp_path / "one"), bufs, bytes(range(240)) * 4, True, 0, 1)
    one = _load_dir(tmp_path / "one")
    assert sorted(one) == sorted([f"{n}_{v}" for n in ("response", "new_challenge") for v in b.VECTORS] +
                                 ["ratio_pairs", "verdict"])
    assert all(a.dtype in (np.float32, np.float64) for a in one.values())
    assert one["verdict"].tolist() == [1.0] and one["ratio_pairs"].tolist() == list(range(240)) * 4
    for name, t, offs in bufs:
        for v, (o, cnt, sz) in enumerate(offs):
            idx = b.dump_sample(cnt, v)
            assert len(idx) == min(cnt, b.DUMP_ELEMENTS) and (np.diff(idx) > 0).all()
            assert np.array_equal(idx, b.dump_sample(cnt, v))
            assert np.array_equal(one[f"{name}_{b.VECTORS[v]}"], t[o:o + cnt * sz].view(cnt, sz).numpy()[idx])
    # at the metric's 2^22 every vector but beta_g2 is sampled: at most 64 MB of float32 in all
    assert b.DUMP_ELEMENTS * (48 + 96 + 48 + 48 + 96 + 192 + 96 + 96) * 4 < 64 << 20
    # two ranks, each holding only its shard, write the same files
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.start_processes(_dump_worker, args=(2, port, str(tmp_path / "two")), nprocs=2, start_method="spawn")
    two = _load_dir(tmp_path / "two")
    assert sorted(two) == sorted(one) and all(np.array_equal(one[k], two[k]) for k in one)


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_round(tmp_path):
    """At 2^10 every element is dumped: the response and new challenge are the C++ oracle's contribution 'bench-1' to
    the challenge 'bench-0', and the dumped (s, sx) pairs satisfy sx = tau * s."""
    import coracle as O
    import pyref as R
    b = _load_bench()
    k = 10
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--power", str(k), "--steps", "2", "--no-e2e",
                        "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    assert json.loads(p.stdout)["steps"] == 2
    got = _load_dir(tmp_path)
    cv = R.BLS12_377
    prm = R.Phase1Parameters(cv, k, 256)
    k0, k1 = b.keys(b"bench-0"), b.keys(b"bench-1")
    win = (prm.g1_chunk_size, prm.other_chunk_size, 0)
    chal = O.phase1_computation(0, bytes(R.phase1_initialization(prm, False)), prm.get_length(False), False, False, 3,
                                *win, *k0)
    want = {"response": O.phase1_computation(0, chal, prm.get_length(True), False, True, 3, *win, *k1),
            "new_challenge": O.phase1_computation(0, chal, prm.get_length(False), False, False, 3, *win, *k1)}
    from snark_setup_b200 import sharding
    n = 1 << k
    for name, compressed in (("response", True), ("new_challenge", False)):
        for v, (o, cnt, sz) in enumerate(sharding.vector_offsets(2 * n - 1, n, compressed)):
            rows = np.frombuffer(want[name][o:o + cnt * sz], dtype=np.uint8).reshape(cnt, sz)
            assert np.array_equal(got[f"{name}_{b.VECTORS[v]}"], rows), (name, v)
    assert got["verdict"].tolist() == [1.0]
    pairs = got["ratio_pairs"].astype(np.uint8).tobytes()
    tau = k0[0] * k1[0] % cv.r
    o = 0
    for grp, usz in ((0, 96), (1, 192), (0, 96), (0, 96)):
        s_, sx = pairs[o:o + usz], pairs[o + usz:o + 2 * usz]
        assert O.apply_powers(0, grp, s_, False, 3, False, 1, powers=[tau]) == sx
        o += 2 * usz
