"""The C-ABI library loads on a GPU-less box, exports every symbol include/gpushare_b200.h declares,
its structs have the layout the ctypes binding assumes, and device entry points FAIL LOUDLY (negative
status, never a CPU fallback) when there is no driver."""
import ctypes as C
import os
import re
import subprocess

import pytest

from gpushare_device_plugin_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gpushare_b200.h")


def header_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gsb_[a-z_0-9]+)\s*\(", src)))


def test_header_binding_and_library_agree():
    declared = header_functions()
    assert declared == sorted(_abi.SYMBOLS)
    out = subprocess.run(["nm", "-D", "--defined-only", _abi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r" T (gsb_[a-z_0-9]+)", out)))
    assert exported == declared
    assert _abi.lib.gsb_abi_version() == _abi.GSB_ABI_VERSION


def test_no_hard_dependency_on_cuda_or_nvml_libraries():
    out = subprocess.run(["readelf", "-d", _abi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    needed = re.findall(r"NEEDED.*\[(.*?)\]", out)
    assert not any("libcuda" in n or "nvidia-ml" in n or "cudart" in n for n in needed), needed


def test_struct_layouts_match_the_header(tmp_path):
    prog = tmp_path / "layout.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gpushare_b200.h"\n'
                    "int main(void){\n"
                    'printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(gsb_device_info), sizeof(gsb_probe_cfg), '
                    "sizeof(gsb_probe_result), sizeof(gsb_cycle_result), sizeof(gsb_event), sizeof(gsb_pod), "
                    "sizeof(gsb_allocate_ctx), sizeof(gsb_health_stats));\n"
                    'printf("%zu %zu %zu %zu %zu\\n", offsetof(gsb_device_info,total_bytes), offsetof(gsb_probe_result,kernel_ns), '
                    "offsetof(gsb_cycle_result,probe), offsetof(gsb_pod,gpu_idx), offsetof(gsb_allocate_ctx,slices));\n"
                    "return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(prog)], check=True)
    a, b = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    assert [int(x) for x in a.split()] == [C.sizeof(t) for t in (_abi.DeviceInfo, _abi.ProbeCfg, _abi.ProbeResult,
                                                                  _abi.CycleResult, _abi.Event, _abi.Pod,
                                                                  _abi.AllocateCtx, _abi.HealthStats)]
    assert [int(x) for x in b.split()] == [_abi.DeviceInfo.total_bytes.offset, _abi.ProbeResult.kernel_ns.offset,
                                           _abi.CycleResult.probe.offset, _abi.Pod.gpu_idx.offset,
                                           _abi.AllocateCtx.slices.offset]


def test_library_carries_sm100a_code_only():
    out = subprocess.run(["cuobjdump", "-lelf", _abi.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    archs = set(re.findall(r"sm_\d+a?", out.stdout))
    assert archs == {"sm_100a"}, archs


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="this box has a GPU")
def test_device_entry_points_fail_loudly_without_a_driver():
    rc = _abi.lib.gsb_init()
    assert rc == _abi.GSB_ERR_LIBRARY_NOT_FOUND
    assert "could not load" in _abi.last_error()
    n = C.c_uint32(7)
    assert _abi.lib.gsb_device_count(C.byref(n)) == _abi.GSB_ERR_NOT_INITIALIZED
    info = _abi.DeviceInfo()
    assert _abi.lib.gsb_device_info_get(0, C.byref(info)) == _abi.GSB_ERR_NOT_INITIALIZED
    res, cfg = _abi.ProbeResult(), _abi.ProbeCfg(op=_abi.GSB_OP_VERIFY)
    assert _abi.lib.gsb_probe(0, C.byref(cfg), C.byref(res)) == _abi.GSB_ERR_NOT_INITIALIZED
    assert res.status == _abi.GSB_ERR_NOT_INITIALIZED
    arena = C.c_uint64(0)
    assert _abi.lib.gsb_arena_create(0, 0, 0, C.byref(arena)) == _abi.GSB_ERR_NOT_INITIALIZED
    cyc = _abi.CycleResult()
    assert _abi.lib.gsb_cycle(0, 0, 0, 1, 0, None, 0, C.byref(cyc)) == _abi.GSB_ERR_NOT_INITIALIZED
    assert _abi.lib.gsb_health_start(0, 0) == _abi.GSB_ERR_NOT_INITIALIZED
    with pytest.raises(_abi.GsbError):
        _abi.check(rc, "gsb_init")


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "gpushare_device_plugin_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cc", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text and '"oracle/' not in text, f


def test_plain_c99_client_sees_the_reference_bytes(tmp_path):
    """tests/native/c_client.c is what a cgo binding looks like from the C side: strict C99, no C++ types, caller
    buffers. Its printed results are held against the golden vectors and the oracle."""
    from oracle import wire_oracle as wo
    exe = tmp_path / "c_client"
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                    "-o", str(exe), os.path.join(ROOT, "tests", "native", "c_client.c"),
                    "-L", os.path.dirname(_abi.LIB_PATH), "-lgpushare_b200",
                    "-Wl,-rpath," + os.path.dirname(_abi.LIB_PATH)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    line = {l.split(" ", 1)[0]: l.split(" ", 1)[1] for l in out if l.split(" ", 1)[0] != "allocate"}
    allocs = [l.split(" ") for l in out if l.startswith("allocate ")]
    u0, u1 = "GPU-fef8089b-4820-abfc-e83e-94318197576e", "GPU-fef8089c-4820-abfc-e83e-94318197576f"
    assert line["abi"] == str(_abi.GSB_ABI_VERSION) and line["slices"] == "179 183359 0"
    assert line["fake"] == f"46 {wo.generateFakeDeviceID(u0, 178)}" and line["real"] == f"40 {u0}"
    assert line["small-buffer"] == "buffer too small" and line["xid"] == "1 1 1 0 0"
    devs = [[wo.generateFakeDeviceID(u, j), wo.Unhealthy if (u, j) == (u0, 1) else wo.Healthy] for u in (u0, u1) for j in range(3)]
    want = wo.marshal_ListAndWatchResponse(devs)
    assert line["lw"] == f"{len(want)} {want.hex()}" and line["lw179"] == "10451"
    want = wo.marshal_RegisterRequest(wo.Version, wo.serverSockName, wo.resourceName)
    assert line["register"] == f"{len(want)} {want.hex()}"
    pods = [{"metadata": {"name": f"pod-0{i}", "namespace": "default", "uid": f"uid-{i}",
                          "annotations": {wo.EnvResourceIndex: idx, wo.EnvResourceAssumeTime: t, wo.EnvAssignedFlag: "false"}},
             "spec": {"nodeName": "n", "containers": [{"resources": {"limits": {wo.resourceName: "4"}}}]},
             "status": {"phase": "Pending"}} for i, (idx, t) in enumerate([("3", "20"), ("1", "10")])]
    dev_map = {u0: 3, u1: 1}
    envs, pod = wo.Allocate([["a", "b", "c", "d"]], pods, "n", dev_map, 179, wo.GiBPrefix, False)
    assert pod["metadata"]["name"] == "pod-01"
    assert allocs[0][1:6] == ["1", "pod", "1", "req", "4"] and allocs[0][6] == wo.marshal_AllocateResponse(envs).hex()
    envs, pod = wo.Allocate([["a", "b", "c", "d"]], pods[:1], "n", dev_map, 179, wo.GiBPrefix, False)
    assert allocs[1][1:6] == ["1", "pod", "0", "req", "4"] and allocs[1][6] == wo.marshal_AllocateResponse(envs).hex()
    want = wo.marshal_AllocateResponse(wo.buildErrResponse([["a", "b", "c", "d"]], 4, wo.GiBPrefix, 179))
    assert line["err"] == f"0 {want.hex()}"
    want = wo.patchPodAnnotationSpecAssigned(1_700_000_000_000_000_000).decode()
    assert line["patch"] == f"{len(want)} {want}"
    assert line["device_count"] == "not initialized"  # no silent stand-in for a missing driver


def test_event_queue_and_lifecycle_under_concurrency(tmp_path):
    """tests/native/health_stress.cc: inject / wait / stop from many threads and the lifecycle entry points racing
    each other, with no device the library can use (on a GPU box CUDA_VISIBLE_DEVICES hides them, so no prober adds
    events of its own). Every injected event is delivered exactly once; nothing crashes.
    (tools/sanitize.sh runs the same program against a TSan-instrumented build of the library.)"""
    exe = tmp_path / "health_stress"
    subprocess.run(["g++", "-O1", "-std=c++17", "-pthread", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "native", "health_stress.cc"), "-L", os.path.dirname(_abi.LIB_PATH),
                    "-lgpushare_b200", "-Wl,-rpath," + os.path.dirname(_abi.LIB_PATH)], check=True)
    out = subprocess.run([str(exe), "1"], capture_output=True, text=True, timeout=60,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert out.returncode == 0, out.stdout + out.stderr
    f = dict(zip(out.stdout.split()[::2], map(int, out.stdout.split()[1::2])))
    assert f["injected"] == f["received"] > 1000 and f["lifecycle"] > 10 and f["stopped"] > 10


def test_shipped_kernels_move_data_with_tma_bulk_copies():
    """SASS of the in-tree library: every dynamic-schedule and static TMA kernel (the AUTO choices) stages its loads
    with UBLKCP (cp.async.bulk, global -> shared) completed on an mbarrier (SYNCS...TRYWAIT); the LDGSTS ring is the
    cp.async variant; DIRECT has neither. Guards the data path against silently degrading to plain loads."""
    out = subprocess.run(["cuobjdump", "-sass", _abi.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0 or "Function" not in out.stdout:
        pytest.skip("cuobjdump unavailable")
    fns, name = {}, None
    for line in out.stdout.splitlines():
        if "Function :" in line:
            name = line.split("Function :", 1)[1].strip()
            fns[name] = []
        elif name and "/*" in line:
            fns[name].append(line)
    def has(fn, mnemonic):
        return any(mnemonic in l for l in fns[fn])
    dyn = [f for f in fns if "probe_bulk_dyn" in f]
    static = [f for f in fns if "probe_bulk" in f and "dyn" not in f and "warp" not in f]
    cpasync = [f for f in fns if "probe_cpasync" in f]
    direct = [f for f in fns if "probe_direct" in f]
    assert len(dyn) >= 3 and len(static) >= 3 and cpasync and direct
    for f in dyn + static:
        loads = "ILi1E" not in f  # OP is the first template argument: 1 = FILL (stores only, nothing to stage in)
        if loads:
            assert has(f, "UBLKCP.S.G") and has(f, "SYNCS.PHASECHK"), f
    for f in cpasync:
        assert has(f, "LDGSTS") and not has(f, "UBLKCP"), f
    for f in direct:
        assert not has(f, "UBLKCP") and not has(f, "LDGSTS"), f
