"""N>1 plumbing of bench.py on CPU: world_size-2 gloo — barrier, max-over-ranks, rank-0-only
reporting, and the reference arm's "rank 0 alone works" rule. The path itself does not shard
(replicas only), so there is no data-path collective to test."""
import json
import os
import socket
import subprocess
import sys

from tests.ref_answers import recorded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import json, os, sys
sys.path.insert(0, %r)
import bench
rank, world, local, dist = bench.dist_setup(2)
assert world == 2 and dist is not None and dist.get_backend() == "gloo"
bench.barrier_sync(dist, local)
m = bench.allmax(dist, local, 10.0 + rank)        # max over ranks of a per-rank timing
s = bench.allmax(dist, local, 5.0 - rank)
bench.barrier_sync(dist, local)
import time
bench.aligned_start(dist, local)                  # every rank leaves at one agreed instant of the host's monotonic clock
left = time.monotonic_ns() / 1e6
skew = bench.allmax(dist, local, left) + bench.allmax(dist, local, -left)   # max - min over ranks, ms
if rank == 0:
    print(json.dumps({"max": m, "max2": s, "world": world, "start_skew_ms": skew}))
dist.destroy_process_group()
''' % ROOT


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def launch(code_or_args, extra_env=None):
    port = free_port()
    procs = []
    for rank in range(2):
        # no GPU in view: dist_setup takes NCCL and one GPU per rank wherever CUDA is available
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES="", **(extra_env or {}))
        procs.append(subprocess.Popen([sys.executable] + code_or_args, env=env, stdout=subprocess.PIPE,
                                      stderr=subprocess.PIPE, text=True, cwd=ROOT))
    try:
        outs = [p.communicate(timeout=180) for p in procs]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
                p.wait()
    return procs, outs


def test_world_size_2_gloo_max_over_ranks():
    procs, outs = launch(["-c", WORKER])
    assert [p.returncode for p in procs] == [0, 0], outs
    line = json.loads(outs[0][0].strip().splitlines()[-1])
    skew = line.pop("start_skew_ms")
    assert line == {"max": 11.0, "max2": 5.0, "world": 2}
    assert 0 <= skew < 5.0, skew  # (sub-0.1 ms on an idle box; the bound only says the ranks did align)
    assert outs[1][0].strip() == ""  # only rank 0 prints


def test_reference_arm_runs_on_rank0_only():
    fake = os.path.join(ROOT, "oracle", "_fake")
    procs, outs = launch(["bench.py", "--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "3"],
                         {"LD_LIBRARY_PATH": fake, "FAKE_NVML_GPUS": "8"})  # an 8-GPU box: the arm must see only 2
    assert [p.returncode for p in procs] == [0, 0], outs
    line = json.loads(outs[0][0].strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["n_gpus"] == 2 and line["details"]["devices_seen"] == 2
    assert line["details"]["fake_devices"] == 358 and line["setup"]["register_calls"] == 179 * 4 + 179 * 6
    ref = json.loads(recorded("ref_inventory_fake.json", ["bench", "--iters", "3", "--warmup", "1", "--gpus", "2"],
                              {"FAKE_NVML_GPUS": "8"}).stdout)
    assert (line["details"]["fake_devices"], line["details"]["lw_bytes"], line["setup"]["register_calls"]) == \
        (ref["n_devices"], ref["lw_len"], ref["register_calls_per_setup"])
    assert set(line["details"]["phases"]["cycle_us"]) >= {"inventory_p50", "health_poll_p50", "cycle_mean"}
    # the arm runs oracle/_ref/ref_inventory where `make -C oracle` could build it from the reference's sources,
    # else the oracle port
    kind = "reference" if os.access(os.path.join(ROOT, "oracle", "_ref", "ref_inventory"), os.X_OK) else "port"
    assert line["metric"] == "inventory+health-probe cycles/sec" and line["cpu_baseline"]["kind"] == kind
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
    assert outs[1][0].strip() == ""
    sys.path.insert(0, ROOT)
    import bench
    assert line["config"] == bench.shared_config(2)  # the very object our own arm prints: same config, key for key


def test_reference_arm_falls_back_to_the_oracle_port_when_the_built_reference_is_missing():
    """`--impl reference` must not die if oracle/_ref (built from the reference's nvml_dl.c where /root/reference exists)
    did not travel: the oracle port — pynvml + oracle/wire_oracle.py — runs the same phases; kind says which one ran."""
    fake = os.path.join(ROOT, "oracle", "_fake")
    env = dict(os.environ, LD_LIBRARY_PATH=fake, FAKE_NVML_GPUS="8", GSB_BENCH_FORCE_PORT="1")
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "4", "--steps", "3", "--warmup", "3",
                          "--no-allocate"], env=env, capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert out.returncode == 0, out.stderr[-800:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == "port" and line["value"] > 0
    d = line["details"]
    assert (d["devices_seen"], d["fake_devices"], d["lw_bytes"]) == (4, 716, 41804)
    assert line["setup"]["register_calls"] == sum(179 * (1 + 2 * (g + 1) + 1) for g in range(4))  # same quadratic scan
