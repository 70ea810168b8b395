"""Pins the oracle itself (CPU): the numpy and C restatements of the probe spec against the committed
golden vectors and against each other; the answers of the C restatement of the reference's NVML path
(linked with the reference's own nvml_dl.c) against a fake libnvidia-ml with 8 synthetic B200s, as
recorded in tests/golden/ref_inventory_fake.json, against the pure-Python restatement of getDevices +
gogo marshal."""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from gpushare_device_plugin_b200 import _abi
from oracle import probe_oracle as po
from oracle import wire_oracle as wo
from tests.ref_answers import recorded

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "probe_pattern.json")))


def test_mix32_is_murmur3_finaliser():
    got = po.mix32(np.array([0, 1, 0xFFFFFFFF], dtype=np.uint32))
    assert [int(v) for v in got] == [GOLD["mix32"]["0"], GOLD["mix32"]["1"], GOLD["mix32"]["4294967295"]]
    assert GOLD["mix32"]["1"] == 0x514E28B7 and GOLD["mix32"]["4294967295"] == 0x81F16F39  # published values


@pytest.mark.parametrize("v", GOLD["words"], ids=lambda v: f"w{v['first_word']}-s{v['seed']}")
def test_pattern_words_golden(v, c_oracle):
    want = np.array(v["lanes"], dtype=np.uint32)
    assert np.array_equal(po.pattern(v["first_word"], 4, v["seed"]), want)
    out = np.empty((4, 4), dtype=np.uint32)
    c_oracle.po_pattern(C.c_uint64(v["first_word"]), C.c_uint64(4), C.c_uint32(v["seed"]), out.ctypes.data_as(C.c_void_p))
    assert np.array_equal(out, want)


@pytest.mark.parametrize("v", GOLD["windows"], ids=lambda v: f"w{v['first_word']}+{v['n_words']}")
def test_window_checksums_golden(v, c_oracle):
    p = po.pattern(v["first_word"], v["n_words"], v["seed"])
    assert po.checksums(p) == (v["checksum_xor"], v["checksum_sum"])
    res = (C.c_uint32 * 2)()
    c_oracle.po_pattern_checksums(C.c_uint64(v["first_word"]), C.c_uint64(v["n_words"]), C.c_uint32(v["seed"]), res)
    assert (res[0], res[1]) == (v["checksum_xor"], v["checksum_sum"])
    # verify() on clean data reports exactly the checksums and no mismatch; a flipped bit is found
    r = po.verify(p, v["first_word"], v["seed"])
    assert (r["mismatch_words"], r["checksum_xor"]) == (0, v["checksum_xor"])
    q = p.copy()
    q[v["n_words"] // 2, 1] ^= np.uint32(1 << 7)
    r = po.verify(q, v["first_word"], v["seed"])
    assert (r["mismatch_words"], r["mismatch_bits"]) == (1, 1)
    assert r["first_bad_offset"] == (v["first_word"] + v["n_words"] // 2) * 16
    res4 = (C.c_uint64 * 4)()
    c_oracle.po_verify.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_void_p]
    first = c_oracle.po_verify(q.ctypes.data_as(C.c_void_p), v["first_word"], v["n_words"], v["seed"], res4)
    assert (first, res4[2], res4[3]) == (v["first_word"] + v["n_words"] // 2, 1, 1)
    assert (res4[0], res4[1]) == (r["checksum_xor"], r["checksum_sum"])


def test_checksums_are_linear_over_disjoint_windows():
    whole = po.checksums(po.pattern(1000, 5000, 3))
    parts = [po.checksums(po.pattern(a, b - a, 3)) for a, b in ((1000, 1001), (1001, 3333), (3333, 6000))]
    assert po.fold(parts) == whole
    assert po.checksums(po.pattern(5, 0, 1)) == (0, 0)


def test_seeds_never_collide_and_addresses_are_unique():
    a, b = po.pattern(0, 4096, 1), po.pattern(0, 4096, 2)
    assert (a != b).all()  # a word that kept an old generation always mismatches
    assert len({tuple(r) for r in po.pattern((1 << 32) - 2048, 4096, 9)}) == 4096  # across the 2^32 word boundary


def run_ref(args, env_extra):
    return recorded("ref_inventory_fake.json", args, env_extra)


class TestReferenceRestatement:
    def test_without_nvml_it_reports_the_reference_error(self):
        out = run_ref(["inventory"], None)
        assert out.returncode == 12 and "could not load NVML library" in out.stderr  # bindings.go:60-66
        assert _abi.lib.gsb_strerror(_abi.GSB_ERR_LIBRARY_NOT_FOUND).decode() in out.stderr  # the product says the same

    @pytest.mark.parametrize("n", [1, 2, 8])
    def test_inventory_matches_python_restatement(self, n):
        out = run_ref(["inventory", "--lw-out"], {"FAKE_NVML_GPUS": str(n)})
        assert out.returncode == 0, out.stderr
        j = json.loads(out.stdout)
        assert (j["n_gpus"], j["gpu_memory"], j["n_devices"]) == (n, 179, 179 * n)
        devs, names, mem = wo.getDevices([{"uuid": d["uuid"], "path": d["path"], "memory_mib": d["memory_mib"]}
                                          for d in j["devices"]])
        lw = wo.marshal_ListAndWatchResponse(devs)
        assert mem == 179 and hashlib.sha256(lw).hexdigest() == out.lw_sha256
        assert len(lw) == j["lw_len"] == {1: 10451, 2: 20902, 8: 83608}[n]  # SURVEY.md §8(a) a7
        assert names == {d["uuid"]: d["minor"] for d in j["devices"]}
        assert all(d["memory_mib"] == 183359 and d["total_bytes"] == 192265846784 for d in j["devices"])

    def test_mib_unit(self):
        out = run_ref(["inventory", "--unit", "MiB"], {"FAKE_NVML_GPUS": "1"})
        j = json.loads(out.stdout)
        assert j["gpu_memory"] == 183359 and j["n_devices"] == 183359

    def test_health_setup_is_quadratic_like_the_reference(self):
        out = run_ref(["bench", "--iters", "2"], {"FAKE_NVML_GPUS": "8"})
        j = json.loads(out.stdout)
        # per fake device: GetCount + (HandleByIndex + GetUUID) x (gpu index + 1) + RegisterEvents
        want = sum(179 * (1 + 2 * (g + 1) + 1) for g in range(8))
        assert j["register_calls_per_setup"] == want == 15752

    def test_bench_arm_sees_only_the_gpus_it_is_asked_for(self):
        """bench.py --impl reference --gpus N must compare N devices with N devices: --gpus caps GetCount everywhere
        it is asked (getDevices and RegisterEventForDevice's scan), like a node that has N GPUs."""
        for n, lw in ((1, 10451), (2, 20902), (4, 41804)):
            j = json.loads(run_ref(["bench", "--iters", "3", "--warmup", "1", "--gpus", str(n)], {"FAKE_NVML_GPUS": "8"}).stdout)
            assert (j["n_gpus"], j["n_devices"], j["lw_len"]) == (n, 179 * n, lw)
            assert j["register_calls_per_setup"] == sum(179 * (1 + 2 * (g + 1) + 1) for g in range(n))
            assert j["cycle_us"]["mean"] > 0 and j["health_setup_us"]["p50"] > 0
        j = json.loads(run_ref(["inventory", "--gpus", "2"], {"FAKE_NVML_GPUS": "8"}).stdout)
        assert j["n_gpus"] == 2 and len(j["devices"]) == 2


def test_pynvml_twin_of_the_reference_inventory_runs_against_the_fake_nvml():
    """bench.py --impl reference also times the NewDevice getter sequence (nvml.go:297-359) through pynvml as a
    sanity bound (SURVEY §8(d)); here the same function against oracle/_fake's libnvidia-ml stand-in."""
    import subprocess
    import sys
    fake = os.path.join(ROOT, "oracle", "_fake")
    if not os.path.exists(os.path.join(fake, "libnvidia-ml.so.1")):
        pytest.skip("oracle/_fake not built")
    env = dict(os.environ, LD_LIBRARY_PATH=fake, FAKE_NVML_GPUS="8", PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, "-c", "import bench, json; print(json.dumps(bench.pynvml_twin(3)))"],
                         capture_output=True, text=True, env=env, cwd=ROOT, timeout=120)
    r = json.loads(out.stdout.strip().splitlines()[-1])
    assert r.get("n_gpus") == 8 and r["iters"] == 3 and r["inventory_us_p50"] > 0, (r, out.stderr[-500:])


def test_product_pattern_header_on_the_host_equals_both_oracles(tmp_path):
    """csrc/gsb_pattern.h is what the sm_100a kernels include; it also compiles for the host. Here it is held against
    the numpy oracle, the golden fixture and (through the numpy oracle's own test) the C oracle — a divergence of the
    product's pattern from its specification shows up on the GPU-less builder, not first on a B200."""
    exe = tmp_path / "pattern_host"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-O1", "-I",
                    os.path.join(ROOT, "gpushare_device_plugin_b200", "csrc"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "native", "pattern_host.c")], check=True)
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "probe_pattern.json")))
    out = subprocess.run([str(exe), "mix", *gold["mix32"].keys()], capture_output=True, text=True, check=True).stdout.split()
    assert [int(x) for x in out] == list(gold["mix32"].values())
    for w in gold["words"]:
        out = subprocess.run([str(exe), "word", str(w["first_word"]), str(len(w["lanes"])), str(w["seed"])],
                             capture_output=True, text=True, check=True).stdout
        assert [[int(x) for x in ln.split()] for ln in out.splitlines()] == w["lanes"]
    rng = np.random.default_rng(7)
    for _ in range(12):  # random windows, including word indices beyond 2^32 (the hi32 term) and seeds up to 2^32-1
        first = int(rng.integers(0, 1 << 34)) if rng.random() < 0.7 else (1 << 32) - 3
        n, seed = int(rng.integers(1, 300)), int(rng.integers(0, 1 << 32))
        out = subprocess.run([str(exe), "word", str(first), str(n), str(seed)], capture_output=True, text=True, check=True).stdout
        got = np.array([[int(x) for x in ln.split()] for ln in out.splitlines()], dtype=np.uint32)
        assert np.array_equal(got, po.pattern(first, n, seed).reshape(-1, 4))
