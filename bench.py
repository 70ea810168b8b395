#!/usr/bin/env python
"""bench.py — inventory + health-probe cycles/s (BASELINE.json's metric) on N B200s of one node.

One step = one cycle of ONE device through the C ABI call `gsb_cycle` (include/gpushare_b200.h): identity + total
(NVML's (re)start-time answer, identity re-validated against the CUDA driver every cycle — the reference asks NVML
once per plugin start too, server.go:39) -> slice count -> S fake devices -> ListAndWatchResponse bytes ->
VERIFY_REFILL launch of the sm_100a probe kernel over this cycle's window of the arena -> verdict folded into
Health. The path does not shard (SURVEY.md §8(e)): under torchrun every rank is an independent replica on its own
GPU, no data-path collective; value = device-cycles all ranks completed / max-over-ranks time ("scaling": "weak").

Headline workload (config.workload): steady state, W = 1 GiB (= one advertised aliyun.com/gpu-mem slice) rotating
over an arena of ALL allocatable HBM (~177.7 GiB), so no window is ever L2-resident.

  value      cycles/s from the CUDA-event time of the probe launches ONLY (arena resident in HBM; excludes
             inventory, encode and every host cost — it is the roofline's companion, not a speed-up claim)
  e2e        cycles/s from host wall time around the gsb_cycle calls (identity check, encode, launch, completion
             wait, result read-back from pinned host memory): the number to hold against `--impl reference`;
             mean-based `value` plus p50/p99 per step
  roofline   algorithmic bytes 2*W per launch / mean CUDA-event duration, vs MEASURED_PEAKS.json hbm_gbs
  setup      what is paid once per plugin start and is NOT in any cycle: ours = gsb_init (dlopen, nvmlInit, cuInit,
             first NVML inventory) + arena (VMM map of all allocatable HBM + FILL); the reference's = nvmlInit +
             first getDevices + watchXIDs' registration loop. Reported on both arms, timed in neither.
  legs (same run, outside the headline's timed region, each with its own numbers):
    live_nvml   the round-1 cycle: a fresh NVML UUID/minor/MemoryInfo query every cycle (GSB_INVENTORY_LIVE)
    full_walk   W = the whole arena, one launch
    transient   the tenant-safe daemon default: no standing arena; allocate W -> FILL -> VERIFY -> free per cycle
    node_cycle  ONE process, all N devices of the run through gsb_cycle_all (what the daemon does; BASELINE
                config 3): rank 0 alone, after every rank has released its arena
  cpu_baseline / --impl reference --gpus N: the reference's NVML call sequence (oracle/_ref/ref_inventory, built
             with the reference's own nvml_dl.c) on this box's host cores, 1 thread — the reference is sequential by
             construction (nvidia.go:59) and budgeted 1 CPU (device-plugin-ds.yaml:34-40) — over the first N GPUs:
             one cycle = getDevices (N x 11 NVML getters + fan-out + marshal) + one WaitForEvent(0) on the standing
             event set. It never touches HBM.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GiB = 1 << 30
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "ref_inventory")
METRIC = "inventory+health-probe cycles/sec"
UNIT = "cycles/s"
WORKLOAD = ("1xB200-per-rank inventory+health cycle: ListAndWatch inventory of 1-GiB aliyun.com/gpu-mem slices "
            "(BASELINE.json configs[1]) + health check, steady state")
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback


def shared_config(n_gpus: int) -> dict:
    """The `config` object BOTH arms print, key for key and value for value (the reference arm runs "on your arm's
    config"); everything arm-specific is under `details`."""
    return {"workload": WORKLOAD, "gpus": n_gpus, "memory_unit": "GiB",
            "slices": "floor(floor(nvmlMemory_t.total / 2^20) / 1024) per GPU (179 on a B200), one fake device per slice",
            "cycle": "one cycle of one device = inventory (identity + total -> slices -> fake devices -> ListAndWatchResponse "
                     "bytes) + one health check; N devices: N such cycles per node cycle",
            "l2_policy": "ours: inputs larger than L2 — the 1 GiB probe window rotates over an arena of all allocatable HBM, no "
                         "flush needed; reference: touches no HBM",
            "value_timing": "ours: `value` = CUDA events around each probe launch on the launching stream, the KERNEL ONLY (no "
                            "inventory, encode or host cost: value / reference.value is not a speed-up), `e2e` = host wall time "
                            "around the C-ABI calls, the like-for-like figure; reference: `value` = `e2e` = host monotonic clock "
                            "around each cycle inside the C binary",
            "setup": "once-per-plugin-start work (ours: gsb_init + arena map + FILL; reference: nvmlInit + first getDevices + "
                     "event-set registration) is reported under `setup` on both arms and is in no timed cycle"}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + throttle reasons of one GPU sampled DURING the timed region: every 10 ms by a thread, plus one
    explicit sample right after the region starts and one right before it ends (the headline region can be as short
    as 20 x 0.34 ms; the GPU has been under the same load since the warm-up steps).

    Sampled in-process through NVML (two calls per sample: nvmlDeviceGetClockInfo and
    nvmlDeviceGetCurrentClocksEventReasons — the same values `nvidia-smi --query-gpu=clocks.sm,
    clocks_event_reasons.*` prints). A separate `nvidia-smi -lms` process per rank was measurably
    perturbing the thing being timed: its polling contends with the cycle's own NVML memory query on
    the driver lock (inventory 6.6 us -> 50 us at N=1, -> 1.6 ms with 8 samplers; profiles/README.md).
    Falls back to nvidia-smi only if pynvml is unusable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int, period_s: float = 0.01):
        self.idx, self.period = gpu_index, period_s
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        self.source = "nvml"
        self._nv = None
        self._lock = threading.Lock()

    def _nvml_setup(self):
        import pynvml
        pynvml.nvmlInit()
        self._nv = pynvml
        self._h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        self._get_reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

    def sample_now(self):
        """One sample from the calling thread (used to bracket the timed region). Never raises."""
        try:
            if self._nv is None:
                self._nvml_setup()
            with self._lock:
                self.sm.append(float(self._nv.nvmlDeviceGetClockInfo(self._h, self._nv.NVML_CLOCK_SM)))
                mask = int(self._get_reasons(self._h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
        except Exception:  # noqa: BLE001
            pass

    def _run_nvml(self):
        if self._nv is None:
            self._nvml_setup()
        while not self._stop.is_set():
            self.sample_now()
            self._stop.wait(self.period)

    def _run_smi(self):
        self.source = "nvidia-smi"
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx)],
                               capture_output=True, text=True)
            p = [x.strip() for x in o.stdout.split(",")]
            if len(p) >= 6:
                try:
                    self.sm.append(float(p[0]))
                    self.max_mhz = float(p[1])
                except ValueError:
                    pass
                self.reasons.update(n for n, v in zip(names, p[2:6]) if v.lower().startswith("active"))
            self._stop.wait(self.period)

    def start(self):
        try:
            self._nvml_setup()
        except Exception:  # noqa: BLE001
            self._nv = None

        def run():
            try:
                if self._nv is None:
                    raise RuntimeError("pynvml unusable")
                self._run_nvml()
            except Exception:
                try:
                    self._run_smi()
                except Exception:
                    pass
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()

    def stop(self) -> dict:
        self._stop.set()
        if self._t:
            self._t.join(timeout=3)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "samples": len(self.sm), "reasons": sorted(self.reasons), "source": self.source,
                "period_ms": int(self.period * 1000)}


def dist_setup(n_gpus: int):
    """torch.distributed is plumbing only: barrier + max-over-ranks of the timings."""
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(
        os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    return rank, world, local, dist


def barrier_sync(dist, local):
    """dist.barrier() + torch.cuda.synchronize(): one bracket of a timed region. (At N = 8 the NCCL barrier itself takes
    ~0.85 ms once the ranks arrive together — a one-element all-reduce on a resident tensor measured the same, so it is
    NCCL's latency, not this call's overhead; 0.2 ms at N = 2. bench reports it per rank as closing_barrier_ms.)"""
    if dist is not None:
        import torch
        dist.barrier()
        if torch.cuda.is_available():
            torch.cuda.synchronize(local)


def aligned_start(dist, local):
    """Opening bracket of a timed region: barrier + synchronize, then every rank spins to ONE agreed instant of the
    host's monotonic clock (system-wide on Linux), 1 ms after the latest rank's "now". Ranks leave an NCCL barrier up
    to ~1 ms apart (host wake-up); without this, a rank that left early waits that long at the CLOSING barrier, which
    is 15 % of a 20-step region at N = 8 and says nothing about the K steps."""
    barrier_sync(dist, local)
    if dist is None:
        return
    target_us = allmax(dist, local, float(time.monotonic_ns() // 1000)) + 1000.0
    while time.monotonic_ns() // 1000 < target_us:
        pass


def allmax(dist, local, x: float) -> float:
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}" if torch.cuda.is_available() else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_reference_cycles(iters: int, warmup: int, gpus: int = 0, setup_iters: int = 3) -> dict:
    """oracle/_ref/ref_inventory bench over the first `gpus` GPUs (0 = all): health set-up once
    (RegisterEventForDevice per fake device), then `iters` timed cycles of inventory (11 NVML getters/GPU + fan-out +
    marshal) + one WaitForEvent(0 ms) on the standing event set, on 1 pinned host thread."""
    if not os.access(REF_BIN, os.X_OK) or os.environ.get("GSB_BENCH_FORCE_PORT") == "1":
        # oracle/_ref is built from the reference's own nvml_dl.c where /root/reference exists and travels with the repo;
        # should it be missing, the arm does not die: the oracle PORT (pynvml + oracle/wire_oracle.py) runs the same phases
        return run_reference_cycles_port(iters, warmup, gpus, setup_iters)
    cmd = [REF_BIN, "bench", "--iters", str(iters), "--warmup", str(warmup), "--wait-ms", "0",
           "--setup-iters", str(setup_iters)]
    if gpus:
        cmd += ["--gpus", str(gpus)]
    if subprocess.run(["taskset", "-c", "0", "true"], capture_output=True).returncode == 0:
        cmd = ["taskset", "-c", "0"] + cmd
    out = subprocess.run(cmd, check=True, capture_output=True, text=True, timeout=600)
    return json.loads(out.stdout.strip().splitlines()[-1])


def run_reference_cycles_port(iters: int, warmup: int, gpus: int = 0, setup_iters: int = 3) -> dict:
    """The same phases as oracle/ref_inventory.c, as the oracle PORT: NVML through pynvml (an independent binding of the
    same libnvidia-ml calls), fan-out and gogo marshal through oracle/wire_oracle.py. Single thread. `kind` = "port"."""
    import pynvml as nv
    from oracle import wire_oracle as wo
    t0 = time.perf_counter_ns()
    nv.nvmlInit()
    init_us = (time.perf_counter_ns() - t0) / 1e3

    def soft(fn, *a):  # bindings.go: NOT_SUPPORTED => nil value, not an error
        try:
            return fn(*a)
        except nv.NVMLError:
            return None

    def count():
        n = nv.nvmlDeviceGetCount()
        return min(n, gpus) if gpus else n

    def get_devices():  # nvidia.go:53-89 over nvml.NewDevice (nvml.go:297-359)
        inv = []
        for i in range(count()):
            h = nv.nvmlDeviceGetHandleByIndex(i)
            soft(nv.nvmlDeviceGetName, h)
            uuid = nv.nvmlDeviceGetUUID(h)
            minor = nv.nvmlDeviceGetMinorNumber(h)
            soft(nv.nvmlDeviceGetPowerManagementLimit, h)
            mem = nv.nvmlDeviceGetMemoryInfo(h)
            pci = soft(nv.nvmlDeviceGetPciInfo, h)
            soft(nv.nvmlDeviceGetBAR1MemoryInfo, h)
            soft(nv.nvmlDeviceGetMaxPcieLinkGeneration, h)
            soft(nv.nvmlDeviceGetMaxPcieLinkWidth, h)
            soft(nv.nvmlDeviceGetMaxClockInfo, h, nv.NVML_CLOCK_SM)
            soft(nv.nvmlDeviceGetMaxClockInfo, h, nv.NVML_CLOCK_MEM)
            if pci is not None:
                bus = pci.busId.decode() if isinstance(pci.busId, bytes) else pci.busId
                try:
                    with open(f"/sys/bus/pci/devices/{bus.lower()[4:] if len(bus) > 12 else bus.lower()}/numa_node") as f:
                        f.read()
                except OSError:
                    pass
            uuid = uuid.decode() if isinstance(uuid, bytes) else uuid
            inv.append({"uuid": uuid, "path": f"/dev/nvidia{minor}", "memory_mib": wo.mib_from_bytes(int(mem.total))})
        devs, _, _ = wo.getDevices(inv)
        return devs

    def register_all(devs):  # nvidia.go:101-117 + bindings.go:97-128 (count + linear HandleByIndex/GetUUID scan)
        es = nv.nvmlEventSetCreate()
        calls = 0
        for id_, _health in devs:
            real = wo.extractRealDeviceID(id_)
            n = count()
            calls += 1
            for i in range(n):
                h = nv.nvmlDeviceGetHandleByIndex(i)
                u = nv.nvmlDeviceGetUUID(h)
                calls += 2
                if (u.decode() if isinstance(u, bytes) else u) == real:
                    nv.nvmlDeviceRegisterEvents(h, nv.nvmlEventTypeXidCriticalError, es)
                    calls += 1
                    break
        return es, calls

    t_reg, es, reg_calls, first_inv_us = [], None, 0, 0.0
    for si in range(max(1, setup_iters)):
        a = time.perf_counter_ns()
        devs = get_devices()
        if si == 0:
            first_inv_us = (time.perf_counter_ns() - a) / 1e3
        if es is not None:
            nv.nvmlEventSetFree(es)
        b = time.perf_counter_ns()
        es, reg_calls = register_all(devs)
        t_reg.append((time.perf_counter_ns() - b) / 1e3)
    t_inv, t_wait, t_cyc, lw = [], [], [], b""
    for it in range(-warmup, iters):
        a = time.perf_counter_ns()
        devs = get_devices()
        lw = wo.marshal_ListAndWatchResponse(devs)
        b = time.perf_counter_ns()
        try:
            nv.nvmlEventSetWait_v2(es, 0) if hasattr(nv, "nvmlEventSetWait_v2") else nv.nvmlEventSetWait(es, 0)
        except nv.NVMLError:
            pass  # timeout
        c = time.perf_counter_ns()
        if it >= 0:
            t_inv.append((b - a) / 1e3)
            t_wait.append((c - b) / 1e3)
            t_cyc.append((c - a) / 1e3)
    nv.nvmlEventSetFree(es)

    def dist_of(v):
        v = sorted(v)
        q = lambda f: v[min(len(v) - 1, int(round(f * (len(v) - 1))))]  # noqa: E731
        return {"p10": q(.1), "p50": q(.5), "p90": q(.9), "p99": q(.99), "mean": sum(v) / len(v)}
    return {"mode": "bench", "kind": "port", "iters": iters, "setup_iters": setup_iters, "n_gpus": count(), "gpu_limit": gpus,
            "n_devices": len(devs), "lw_len": len(lw), "wait_ms": 0, "nvml_init_us": init_us, "first_inventory_us": first_inv_us,
            "register_calls_per_setup": reg_calls, "register_rc": 0, "wait_rc": 10,
            "inventory_us": dist_of(t_inv), "health_setup_us": dist_of(t_reg), "health_poll_us": dist_of(t_wait),
            "cycle_us": dist_of(t_cyc), "total_us": sum(t_cyc)}


def reference_phases(r: dict) -> dict:
    return {"cycle_us": {"inventory_p50": r["inventory_us"]["p50"], "health_poll_p50": r["health_poll_us"]["p50"],
                         "cycle_p50": r["cycle_us"]["p50"], "cycle_p99": r["cycle_us"]["p99"], "cycle_mean": r["cycle_us"]["mean"]},
            "setup_once_per_start_us": {"nvml_init": r["nvml_init_us"], "first_inventory": r["first_inventory_us"],
                                        "health_setup_p50": r["health_setup_us"]["p50"],
                                        "register_calls": r["register_calls_per_setup"], "register_rc": r["register_rc"]}}


def pynvml_twin(iters: int) -> dict:
    """SURVEY §8(d): the same NewDevice getter sequence (nvml.go:297-359) through pynvml, as a sanity bound on the
    C restatement's inventory phase — an independent binding over the same libnvidia-ml calls. Never fatal."""
    try:
        import pynvml as nv
        nv.nvmlInit()

        def soft(fn, *a):  # bindings.go: NOT_SUPPORTED => nil value, not an error
            try:
                return fn(*a)
            except nv.NVMLError:
                return None
        times = []
        n = nv.nvmlDeviceGetCount()
        for _ in range(iters):
            t0 = time.perf_counter_ns()
            for i in range(nv.nvmlDeviceGetCount()):
                h = nv.nvmlDeviceGetHandleByIndex(i)
                soft(nv.nvmlDeviceGetName, h)
                soft(nv.nvmlDeviceGetUUID, h)
                soft(nv.nvmlDeviceGetMinorNumber, h)
                soft(nv.nvmlDeviceGetPowerManagementLimit, h)
                soft(nv.nvmlDeviceGetMemoryInfo, h)
                pci = soft(nv.nvmlDeviceGetPciInfo, h)
                soft(nv.nvmlDeviceGetBAR1MemoryInfo, h)
                soft(nv.nvmlDeviceGetMaxPcieLinkGeneration, h)
                soft(nv.nvmlDeviceGetMaxPcieLinkWidth, h)
                soft(nv.nvmlDeviceGetMaxClockInfo, h, nv.NVML_CLOCK_SM)
                soft(nv.nvmlDeviceGetMaxClockInfo, h, nv.NVML_CLOCK_MEM)
                if pci is not None:  # numaNode(busid): one sysfs read (nvml.go:262-295)
                    bus = pci.busId.decode() if isinstance(pci.busId, bytes) else pci.busId
                    try:
                        with open(f"/sys/bus/pci/devices/{bus.lower()[4:] if len(bus) > 12 else bus.lower()}/numa_node") as f:
                            f.read()
                    except OSError:
                        pass
            times.append(time.perf_counter_ns() - t0)
        times.sort()
        return {"n_gpus": n, "iters": iters, "inventory_us_p50": times[len(times) // 2] / 1e3, "inventory_us_min": times[0] / 1e3}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[-200:]}


def cpu_model() -> str:
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


UUIDS8 = ["GPU-%08x-4820-abfc-e83e-9431819757%02x" % (0xfef80890 + i, i) for i in range(8)]


def bench_allocate(impl: str, quick: bool = False) -> dict:
    """p50 Allocate() (BASELINE.json's second metric), SURVEY.md §8(d) configs 4-5, host-only: real grpc over
    a unix socket, a stateful loopback mock apiserver that applies the PATCH, synthetic 8-GPU inventory
    (the RPC never touches a GPU in either implementation). `ours` = nvidia/server.py over the C ABI
    (gsb_allocate) with the pending-pod cache — `ours` = the native daemon gsbd, `ours_py` = the Python front
    end; `reference` = oracle/ref_plugin.py (global lock across I/O, LIST per call, Python codec, synchronous
    log lines)."""
    import logging
    import resource
    import shutil
    from gpushare_device_plugin_b200.testing import socket_dir
    soft, hard = resource.getrlimit(resource.RLIMIT_NOFILE)  # c = 1 024 needs > 2 048 descriptors in the in-process arms
    if soft < hard:
        resource.setrlimit(resource.RLIMIT_NOFILE, (hard, hard))
    logging.getLogger("gpushare").setLevel(logging.WARNING)
    logging.getLogger("gpushare.nvidia").setLevel(logging.WARNING)
    node = "b200-0"
    native_mock = os.path.join(ROOT, "gpushare_device_plugin_b200", "gsb_mock_kube")
    use_native_mock = os.access(native_mock, os.X_OK) and os.environ.get("GSB_BENCH_MOCK", "native") == "native"
    mock_argv = [native_mock] if use_native_mock else [sys.executable, "-m", "gpushare_device_plugin_b200.testing.mock_kube"]
    out = {"impl": impl, "transport": "gRPC (HTTP/2) over a unix socket; the server is the arm under test",
           "mock": ("loopback compiled apiserver stand-in (csrc/daemon/mock_kube.cc)" if use_native_mock else
                    "loopback Python apiserver") + ", own process; clients in a third process",
           "sweep": []}

    def start(n_pods, mod, gsbd_extra=()):
        tmp = socket_dir("gsb-alloc-")
        kube = subprocess.Popen(mock_argv + ["--node", node, "--pods", str(n_pods)] + (["--mod"] if mod else []),
                                stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True, cwd=ROOT)
        url = f"http://127.0.0.1:{int(kube.stdout.readline())}"
        sock = os.path.join(tmp, "aliyungpushare.sock")
        minors = {u: i for i, u in enumerate(UUIDS8)}
        if impl == "ours":  # the native daemon (gsbd): C++ HTTP/2 front end + C ABI, no interpreter on the RPC path
            from gpushare_device_plugin_b200.testing.fake_kubelet import FakeKubelet
            kubelet = FakeKubelet(tmp)
            env = dict(os.environ, NODE_NAME=node, GPUSHARE_PLUGIN_DIR=tmp + "/", GPUSHARE_DUMP_DIR=tmp,
                       GSBD_ALLOW_FAKE_INVENTORY="1")
            env.pop("KUBECONFIG", None)
            proc = subprocess.Popen([os.path.join(ROOT, "gpushare_device_plugin_b200", "gsbd"), "-logtostderr", "--v=5",
                                     "--fake-inventory", "8",  # the DaemonSet's own flags: every glog line is produced
                                     "--kube-api-url", url] + list(gsbd_extra) + os.environ.get("GSBD_EXTRA", "").split(), env=env, stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL)
            kubelet.register_requests.get(timeout=30)
            time.sleep(0.3)  # let the pod informer finish its first LIST + watch (the kubelet calls Allocate much later)

            def stop():
                proc.terminate()
                proc.wait(timeout=10)
                kubelet.stop()
        elif impl == "ours_py":  # the Python front end (nvidia/server.py, grpcio) over the same C ABI
            from gpushare_device_plugin_b200 import device
            from gpushare_device_plugin_b200.nvidia import kubeclient, nvidia, podmanager, server
            podmanager.kubeInit(kubeclient.Clientset(url), node)
            nvidia.gpuMemory, nvidia.metric = 179, "GiB"
            devs = [nvidia.Device(ID=device.fake_device_id(u, j)) for u in UUIDS8 for j in range(179)]
            plugin = server.NewNvidiaDevicePlugin(False, False, False, None, socket=sock, inventory=(devs, minors),
                                                  max_workers=64)
            plugin.Start()
            stop = plugin.Stop
        else:
            from oracle.ref_plugin import RefPlugin
            plugin = RefPlugin(url, node, minors, 179, sock)
            plugin.start()
            stop = plugin.stop

        def close():
            stop()
            kube.stdin.close()
            kube.wait(timeout=10)
            shutil.rmtree(tmp, ignore_errors=True)
        return sock, close

    native_client = os.path.join(ROOT, "gpushare_device_plugin_b200", "gsb_alloc_load")
    out["client"] = "native HTTP/2 client (csrc/daemon/alloc_load.cc), one persistent connection per client thread" \
        if os.access(native_client, os.X_OK) else "grpcio (Python) client threads"

    def load(sock, c, total):  # clients in their own process too; the same generator for every arm
        argv = [native_client] if os.access(native_client, os.X_OK) else \
            [sys.executable, "-m", "gpushare_device_plugin_b200.testing.allocate_load"]
        o = subprocess.run(argv + [sock, str(c), str(total), ",".join(UUIDS8)], capture_output=True, text=True, cwd=ROOT,
                           timeout=900)
        if o.returncode:
            raise RuntimeError(o.stderr[-400:])
        return json.loads(o.stdout.strip().splitlines()[-1])

    # config 4: 64 pending pods, 64 sequential Allocates
    sock, close = start(64, False)
    r = load(sock, 1, 64)
    close()
    out["config4"] = {k: r[k] for k in ("p50_us", "p99_us", "mean_us", "req_per_s", "error_responses")}
    if impl == "ours":  # where the time goes: the same daemon with the pod source stepped back towards the reference's
        out["config4_by_pod_source"] = {"watch_informer (default)": out["config4"]["p50_us"]}
        for label, extra in (("ttl_cache (--pod-informer=false)", ("--pod-informer=false",)),
                             ("list_per_call, as the reference (--pod-informer=false --pod-cache-ttl 0)",
                              ("--pod-informer=false", "--pod-cache-ttl", "0")),
                             ("list_per_call + one lock across the PATCH (--serialize-allocate): the reference's Allocate in compiled code",
                              ("--pod-informer=false", "--pod-cache-ttl", "0", "--serialize-allocate"))):
            sock, close = start(64, False, extra)
            out["config4_by_pod_source"][label] = load(sock, 1, 64)["p50_us"]
            close()
        if not quick:  # and what that lock does to concurrency: config 5 at c = 16, reference behaviour in compiled code
            sock, close = start(1024, True, ("--pod-informer=false", "--pod-cache-ttl", "0", "--serialize-allocate"))
            out["compiled_reference_behaviour_c16"] = {k: v for k, v in load(sock, 16, 256).items()
                                                       if k in ("p50_us", "p99_us", "req_per_s", "error_responses", "requests")}
            close()
    # config 5: 1024 pending pods, concurrency sweep 1..1024 (bounded: max(256, c) requests per point)
    for c in ((1, 16) if quick else tuple(1 << k for k in range(11))):  # SURVEY §8(d) config 5: c = 1, 2, 4, ... 1 024
        sock, close = start(1024, True)
        # each Allocate consumes one of the 1 024 pending pods; the reference arm (~40 req/s) gets a smaller sample
        try:
            r = load(sock, c, 64 if quick else (max(128, c) if impl == "reference" else max(1000, c)))
        except Exception as e:  # noqa: BLE001  one point that cannot run (fd limits, a timeout) must not void the others
            r = {"concurrency": c, "error": str(e)[-300:]}
        close()
        out["sweep"].append(r)
    out["p50_us"] = out["config4"]["p50_us"]
    if impl == "ours":
        ref_row = [v for k, v in out.get("config4_by_pod_source", {}).items() if "serialize-allocate" in k]
        out["p50_context"] = {
            "config4_p50_us": out["p50_us"],
            "compiled_reference_behaviour_config4_p50_us": ref_row[0] if ref_row else None,
            "speedup_vs_compiled_reference_behaviour_c1": (ref_row[0] / out["p50_us"]) if ref_row and out["p50_us"] else None,
            "c16": {"ours_p50_us": next((p["p50_us"] for p in out["sweep"] if p.get("concurrency") == 16 and "p50_us" in p), None),
                    "compiled_reference_behaviour_p50_us": out.get("compiled_reference_behaviour_c16", {}).get("p50_us")},
            "note": "the comparison to quote: the same compiled daemon with the reference's behaviour switched back on "
                    "(--pod-informer=false --pod-cache-ttl 0 --serialize-allocate = LIST per call under one lock held across "
                    "the PATCH, allocate.go:59-60). The `--impl reference` arm's Allocate is a Python port and flatters us "
                    "by the interpreter's cost"}
    return out


def bench_reference(args) -> None:
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return  # rank 0 alone runs the (sequential, single-process) reference path
    cps = max(1, args.ref_cycles_per_step)  # one step = a bounded sample of `cps` reference cycles
    r = run_reference_cycles(args.steps * cps, args.warmup * cps, gpus=args.gpus)
    n = r["n_gpus"]
    mean_us = r["cycle_us"]["mean"]
    value = n * 1e6 / mean_us  # one node cycle covers n devices sequentially
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": mean_us * cps / 1e3,
        "ms_per_device_cycle": mean_us / 1e3 / max(n, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": shared_config(args.gpus),
        "details": {"reference_path": f"one cycle = getDevices over the first {n} GPU(s) (11 NVML getters each + fan-out + gogo "
                                      "marshal, nvidia.go:53-89) + one WaitForEvent(0 ms) on the standing event set "
                                      "(nvidia.go:126); sequential, 1 thread; the reference moves no HBM bytes. The event-set "
                                      "registration (S*N RegisterEventForDevice, nvidia.go:104-117) is once per plugin start and "
                                      "is reported under setup, outside the timed cycles — as our arm's arena set-up is",
                    "devices_seen": n, "fake_devices": r["n_devices"], "lw_bytes": r["lw_len"],
                    "cycles_per_step": cps, "cycles_timed": args.steps * cps,
                    "step": f"one step = a bounded sample of {cps} node cycles (NVML latency on a shared host is too noisy for a "
                            "20-cycle mean: 2.2 ms idle, 4-7 ms beside a polling nvidia-smi); ms_per_step is the whole sample",
                    "phases": reference_phases(r),
                    "pynvml_twin": pynvml_twin(min(args.steps, 50)),
                    "host": f"{cpu_model()}, nproc={os.cpu_count()}"},
        "setup": reference_phases(r)["setup_once_per_start_us"],
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": r.get("kind", "reference"),
                         "sample": f"{args.steps * cps} cycles (+{args.warmup * cps} warm-up) of oracle/_ref/ref_inventory (reference's "
                                   f"nvml_dl.c) over {n} GPU(s), taskset -c 0, {cpu_model()}, nproc={os.cpu_count()}"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "p50_value": n * 1e6 / r["cycle_us"]["p50"], "p50_ms_per_step": r["cycle_us"]["p50"] / 1e3 / max(n, 1)},
        "gpu_launches": 0,
    }
    if not args.no_allocate and int(os.environ.get("WORLD_SIZE", 1)) == 1:  # host-only leg: N = 1 runs only
        try:
            line["allocate"] = bench_allocate("reference", args.quick_allocate)
            line["allocate"]["note"] = ("this arm is the behaviour-faithful Python port (oracle/ref_plugin.py: global lock across "
                                        "I/O, LIST per call, Python codec, synchronous log lines); the language-fair row is our "
                                        "arm's allocate.compiled_reference_behaviour")
        except Exception as e:  # noqa: BLE001
            line["allocate"] = {"error": str(e)}
    print(json.dumps(line))


def pctl(sorted_ns, q):
    return sorted_ns[min(len(sorted_ns) - 1, int(q * len(sorted_ns)))]


def timed_cycles(cyc, steps: int, warmup: int, dist, local, sampler=None, capture=None):
    """W warm-up steps, then exactly `steps` steps bracketed by barrier + synchronize; per-step host times kept.
    `sampler` (clocks) runs from before the warm-up to after the last step; the clock samples kept are those taken
    while the GPU was under this load. `capture(cyc)`, if given, runs once the timed region is closed and before any
    further step, and its result is returned as "captured"."""
    if sampler is not None:
        sampler.start()
    for _ in range(warmup):
        cyc.step()
    if sampler is not None:
        sampler.sm.clear()      # keep only samples taken under load (from the last warm-up step on)
        sampler.sample_now()
    aligned_start(dist, local)
    kernel_ns, inv_ns = 0, 0
    per_step = []
    t0 = time.perf_counter_ns()
    for _ in range(steps):
        ts = time.perf_counter_ns()
        r = cyc.step()
        per_step.append(time.perf_counter_ns() - ts)
        if not r.healthy:
            raise RuntimeError(f"probe reported {r.probe.mismatch_words} mismatching words — unhealthy device")
        kernel_ns += r.probe.kernel_ns
        inv_ns += r.inventory_ns
    # every step ends device-synchronised (gsb_cycle returns after the kernel's results are in host memory), so this
    # is a synchronised end-of-region time on this rank; the closing barrier brackets the region but its own latency
    # and the ranks' exit skew from the OPENING barrier (which a wall clock taken after the closing barrier would add
    # to every rank that started early) are not part of the K steps. MAX over ranks is taken by the caller.
    wall_ns = time.perf_counter_ns() - t0
    barrier_sync(dist, local)
    close_ns = time.perf_counter_ns() - t0 - wall_ns
    captured = capture(cyc) if capture is not None else None
    if sampler is not None:
        # the timed region is over (wall_ns is taken): a few more steps of the same load so that even a 7 ms
        # region is covered by samples taken at this clock/power state
        t_end = time.perf_counter() + 0.06
        while time.perf_counter() < t_end:
            cyc.step()
            sampler.sample_now()
    per_step.sort()
    return {"wall_ns": wall_ns, "closing_barrier_ns": close_ns, "kernel_ns": kernel_ns, "inventory_ns": inv_ns, "launches": steps, "last": r,
            "p50_ms": pctl(per_step, 0.5) / 1e6, "p99_ms": pctl(per_step, 0.99) / 1e6, "max_ms": per_step[-1] / 1e6,
            "captured": captured}


def cycle_outputs(cyc, idx: int, arena: int, window: int) -> dict:
    """What the cycler's last gsb_cycle handed its caller, as arrays for --dump-outputs:
      list_and_watch  the ListAndWatchResponse bytes (float32, one byte per element), the card's UUID in them replaced
                      by GPU-00000000-0000-0000-0000-000000000000 so that runs on different cards compare
      inventory       [total_mib, slices]
      probe           [healthy, mismatch_words, mismatch_bits, checksum_xor, checksum_sum, bytes_walked, window_offset]
      window_sample   (64, 16384) 32-bit lanes of the window the cycle's VERIFY_REFILL rewrote, read back from HBM at
                      64 KiB chunks chosen by a fixed seed
    The window rotates over the arena, so with the same arguments the arrays repeat where the arena has the same size."""
    import numpy as np
    from gpushare_device_plugin_b200 import device
    r, p = cyc.res, cyc.res.probe
    n_win = arena // window if window < arena else 1
    offset = ((cyc.cycle_no - 1) % n_win) * window  # the window gsb_cycle walks for this cycle_no
    chunk = 64 << 10
    starts = np.sort(np.random.default_rng(0).choice(p.bytes_walked // chunk, 64, replace=False)) * chunk
    sample = [np.frombuffer(device.arena_read(idx, offset + int(a), chunk), dtype=np.uint32) for a in starts]
    lw = cyc.list_and_watch_bytes().replace(r.info.uuid, b"GPU-00000000-0000-0000-0000-000000000000")
    return {"list_and_watch": np.frombuffer(lw, dtype=np.uint8).astype(np.float32),
            "inventory": np.array([r.info.total_mib, r.slices], dtype=np.float64),
            "probe": np.array([r.healthy, p.mismatch_words, p.mismatch_bits, p.checksum_xor, p.checksum_sum,
                               p.bytes_walked, offset], dtype=np.float64),
            "window_sample": np.stack(sample).astype(np.float64)}


def node_cycle_leg(device, n: int, steps: int, warmup: int, window: int) -> dict:
    """ONE process, all n devices through gsb_cycle_all (one persistent native thread, primary context and
    non-blocking stream per device; one joined ListAndWatchResponse) — what the daemon does, and what replaces the
    reference's sequential loop nvidia.go:59-86. Arena per device: 8 windows (each 1 GiB window >> the 126 MB L2)."""
    from gpushare_device_plugin_b200 import _abi
    t0 = time.perf_counter()
    device.init()
    arenas = [device.arena_create(i, max_bytes=8 * window, keep_free_bytes=2 * GiB) for i in range(n)]
    setup_s = time.perf_counter() - t0
    node = device.NodeCycler(list(range(n)), window_bytes=window)
    for _ in range(warmup):
        node.step()
    per_step, kern, inv = [], [0] * n, [[] for _ in range(n)]
    t0 = time.perf_counter_ns()
    for _ in range(steps):
        ts = time.perf_counter_ns()
        res = node.step()
        per_step.append(time.perf_counter_ns() - ts)
        for i, r in enumerate(res):
            if not r.healthy:
                raise RuntimeError(f"node cycle: device {i} unhealthy")
            kern[i] += r.probe.kernel_ns
            inv[i].append(r.inventory_ns)
    wall_ns = time.perf_counter_ns() - t0
    per_step.sort()
    out = {"n_gpus": n, "steps": steps, "warmup": warmup, "window_bytes": window, "arena_bytes_per_device": min(arenas),
           "node_cycles_per_s": steps / (wall_ns / 1e9), "device_cycles_per_s": n * steps / (wall_ns / 1e9),
           "step_ms": {"min": per_step[0] / 1e6, "p50": pctl(per_step, 0.5) / 1e6, "p99": pctl(per_step, 0.99) / 1e6,
                       "max": per_step[-1] / 1e6, "mean": wall_ns / 1e6 / steps},
           "kernel_ms_per_cycle_per_device": [round(k / 1e6 / steps, 4) for k in kern],
           "inventory_us_p50_per_device": [round(sorted(v)[len(v) // 2] / 1e3, 2) for v in inv],
           "inventory_us_max_per_device": [round(max(v) / 1e3, 2) for v in inv],
           "aggregate_hbm_gbs": sum(2 * window * steps / (k / 1e9) / 1e9 for k in kern if k),
           "lw_bytes": node.lw_len, "devices_advertised": res[0].slices * n,
           "inventory_policy": "live" if device.get_option(_abi.GSB_OPT_INVENTORY_POLICY) else "snapshot",
           "setup_s": round(setup_s, 3)}
    for i in range(n):
        device.arena_destroy(i)
    device.shutdown()
    return out


def bench_ours(args) -> None:
    rank, world, local, dist = dist_setup(args.gpus)
    host_group = None
    if dist is not None:
        host_group = dist.new_group(backend="gloo")  # host-side barrier for the node-cycle leg: no kernel parked on a GPU
    line_cpu = None
    if world == 1 and not args.no_cpu_baseline:
        # FIRST, before this process owns a CUDA context or any HBM: the same binary, flags and state as
        # `--impl reference --gpus 1`, so the two numbers agree within host noise
        try:
            r = run_reference_cycles(args.cpu_iters, 3, gpus=1)
            line_cpu = {"value": r["n_gpus"] * 1e6 / r["cycle_us"]["mean"], "unit": UNIT, "cores": 1, "kind": r.get("kind", "reference"),
                        "sample": f"{args.cpu_iters} cycles (+3 warm-up) of oracle/_ref/ref_inventory (built with the reference's "
                                  f"nvml_dl.c) over 1 GPU, before this process created a CUDA context: inventory p50 "
                                  f"{r['inventory_us']['p50']} us + poll p50 {r['health_poll_us']['p50']} us per cycle; "
                                  f"set-up once per start {r['health_setup_us']['p50']} us ({r['register_calls_per_setup']} NVML "
                                  f"calls), not in the cycle; taskset -c 0; no HBM traffic",
                        "phases": reference_phases(r)}
        except Exception as e:  # noqa: BLE001
            line_cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": f"failed: {e}"}
    from gpushare_device_plugin_b200 import _abi, device
    if dist is not None:  # make NCCL allocate its buffers BEFORE the arena takes all free HBM
        barrier_sync(dist, local)
        allmax(dist, local, 0.0)
    t_setup = time.perf_counter()
    device.init()
    init_ms = (time.perf_counter() - t_setup) * 1e3
    n_dev = device.device_count()
    idx = local if world > 1 else 0
    if idx >= n_dev:
        raise RuntimeError(f"rank {rank}: device index {idx} but only {n_dev} GPUs visible")
    keep_free = (2 * GiB) if dist is not None else 0
    window = args.window_gib * GiB
    variant = {"auto": 0, "direct": 1, "cpasync": 2, "bulk": 3, "bulkw": 4, "bulkd": 5}[args.variant]
    tr = None
    if not args.no_transient:  # before the standing arena exists: allocate -> fill -> verify -> free per cycle
        trc = device.Cycler(idx, window_bytes=window, variant=variant)
        tr = timed_cycles(trc, args.transient_steps, 3, dist, local)
    t_arena = time.perf_counter()
    arena = device.arena_create(idx, keep_free_bytes=keep_free)
    arena_ms = (time.perf_counter() - t_arena) * 1e3
    peak, peak_src = measured_peak()
    device.set_option(_abi.GSB_OPT_INVENTORY_POLICY, _abi.GSB_INVENTORY_LIVE if args.inventory == "live" else _abi.GSB_INVENTORY_SNAPSHOT)

    sampler = ClockSampler(idx)
    # ---- headline: steady-state rotating window ------------------------------------------------
    cyc = device.Cycler(idx, window_bytes=window, variant=variant)
    capture = (lambda c: cycle_outputs(c, idx, arena, window)) if args.dump_outputs and rank == 0 else None
    head = timed_cycles(cyc, args.steps, args.warmup, dist, local, sampler, capture)
    clocks = sampler.stop()
    last = head["last"]
    snapshot_age_ms = last.snapshot_age_ns / 1e6
    # ---- same run, other legs (each outside the headline's timed region) -----------------------------
    other = _abi.GSB_INVENTORY_SNAPSHOT if args.inventory == "live" else _abi.GSB_INVENTORY_LIVE
    device.set_option(_abi.GSB_OPT_INVENTORY_POLICY, other)
    alt = timed_cycles(cyc, min(args.steps, 100), 3, dist, local)
    device.set_option(_abi.GSB_OPT_INVENTORY_POLICY, _abi.GSB_INVENTORY_SNAPSHOT)
    full = device.Cycler(idx, window_bytes=0, variant=variant)
    fw = timed_cycles(full, args.full_steps, 3, dist, local)
    device.arena_destroy(idx)

    if dist is not None:  # every rank sampled its own GPU: report the slowest median and the union of reasons
        allc = [None] * world
        dist.all_gather_object(allc, clocks, group=host_group)
        meds = [c["sm_mhz"] for c in allc if c and c["sm_mhz"] is not None]
        clocks = dict(clocks, sm_mhz=min(meds) if meds else None,
                      reasons=sorted(set(r for c in allc if c for r in c["reasons"])), ranks=world)
    per_rank = None
    if dist is not None:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, {"wall_ms": round(head["wall_ns"] / 1e6, 3), "p50_ms": round(head["p50_ms"], 4),
                                          "p99_ms": round(head["p99_ms"], 4), "max_ms": round(head["max_ms"], 4),
                                          "closing_barrier_ms": round(head["closing_barrier_ns"] / 1e6, 3)}, group=host_group)
    wall_incl_s = allmax(dist, local, (head["wall_ns"] + head["closing_barrier_ns"]) / 1e9)
    wall_s = allmax(dist, local, head["wall_ns"] / 1e9)
    kern_s = allmax(dist, local, head["kernel_ns"] / 1e9)
    p50_s = allmax(dist, local, head["p50_ms"] / 1e3)
    alt_wall_s = allmax(dist, local, alt["wall_ns"] / 1e9)
    f_wall_s = allmax(dist, local, fw["wall_ns"] / 1e9)
    f_kern_s = allmax(dist, local, fw["kernel_ns"] / 1e9)
    tr_wall_s = allmax(dist, local, tr["wall_ns"] / 1e9) if tr else None
    device.shutdown()  # arena, streams, NVML released on every rank before the one-process node cycle
    if dist is not None:
        dist.barrier(group=host_group)
    node = None
    if rank == 0 and not args.no_node_cycle:
        try:
            node = node_cycle_leg(device, world, args.node_steps, 5, window)
        except Exception as e:  # noqa: BLE001
            node = {"error": str(e)[-300:]}
    if dist is not None:
        dist.barrier(group=host_group)
    if rank != 0:
        return

    units = args.steps * world
    f_units = args.full_steps * world
    achieved = 2 * window * args.steps / (head["kernel_ns"] / 1e9) / 1e9  # this rank's kernel, GB/s
    f_achieved = 2 * arena * args.full_steps / (fw["kernel_ns"] / 1e9) / 1e9
    prof = {}
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            prof = json.load(f)
    except Exception:
        pass
    traffic_src = "profiles/ncu_traffic.json: dram__bytes_read+write of this kernel from an `ncu --set full` capture of the same launch shape; NOT measured in this run"
    kname = {1: "probe_direct", 2: "probe_cpasync", 3: "probe_bulk", 4: "probe_bulk_warp", 5: "probe_bulk_dyn"}[last.probe.variant]
    alt_name = "snapshot" if args.inventory == "live" else "live_nvml"
    line = {
        "metric": METRIC, "value": units / kern_s, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": kern_s * 1e3 / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": shared_config(world),
        "details": {"ours_path": f"{last.slices} slices / {last.lw_len} B ListAndWatchResponse + VERIFY_REFILL HBM probe of a "
                                 f"rotating {args.window_gib} GiB window (one advertised slice) over the whole arena",
                    "window_bytes": window, "arena_bytes": arena, "variant": _abi.VARIANT_NAMES[last.probe.variant],
                    "grid_ctas": last.probe.grid_ctas, "block_threads": last.probe.block_threads,
                    "inventory_policy": args.inventory,
                    "replicas": "one independent replica per GPU, no collective (path does not shard)",
                    "host": f"{cpu_model()}, nproc={os.cpu_count()}"},
        "e2e": {"value": units / wall_s, "unit": UNIT, "ms_per_step": wall_s * 1e3 / args.steps,
                "p50_value": world / p50_s, "p50_ms_per_step": p50_s * 1e3,
                "value_incl_closing_barrier": units / wall_incl_s,
                "h2d_bytes_per_step": 120, "d2h_bytes_per_step": 56,
                "note": "gsb_cycle through ctypes: identity check against the CUDA driver, slices, encode, launch, completion "
                        "wait; h2d = kernel argument block, d2h = gsb_kernel_out written by the last CTA into pinned mapped "
                        "host memory; the ListAndWatch bytes are produced on the host. value = steps / total wall (mean); "
                        "p50_value = from the median step (max over ranks)",
                "inventory_us_per_step": head["inventory_ns"] / 1e3 / args.steps,
                "inventory_source": ("NVML queried inside every cycle" if args.inventory == "live" else
                                     f"NVML's answer from gsb_init (age {snapshot_age_ms:.0f} ms at the last step), identity "
                                     "re-validated per cycle via cuDeviceGetUuid; the reference also asks NVML once per start"),
                "per_step_rank0": {"p50_ms": head["p50_ms"], "p99_ms": head["p99_ms"], "max_ms": head["max_ms"]},
                "timed_region": "per rank: opening barrier + synchronize, then all ranks spin to one agreed instant of the host's "
                                "monotonic clock (start-line alignment), t0, K synchronous steps, t1, closing barrier + "
                                "synchronize, t2. value uses MAX over ranks of (t1 - t0): each step ends device-synchronised, "
                                "so t1 is a synchronised time. value_incl_closing_barrier uses MAX over ranks of (t2 - t0), "
                                "i.e. with the closing barrier's own latency inside (per_rank.closing_barrier_ms)",
                "per_rank": per_rank},
        "gpu_launches": head["launches"] * world,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": prof.get("window_1gib_dram_bytes_per_launch"), "traffic_source": traffic_src,
                     "kernel": kname + "<VERIFY_REFILL>",
                     "algorithmic_bytes_per_launch": 2 * window, "peak_source": peak_src},
        "setup": {"once_per_start_ms": {"gsb_init (dlopen, nvmlInit, cuInit, first NVML inventory)": round(init_ms, 1),
                                        "arena (VMM map of all allocatable HBM + FILL of every byte)": round(arena_ms, 1)},
                  "note": "not in any timed cycle; the reference arm reports its own once-per-start work the same way"},
        alt_name: {"e2e_value": min(args.steps, 100) * world / alt_wall_s, "unit": UNIT, "steps": min(args.steps, 100),
                   "inventory_us_per_step": alt["inventory_ns"] / 1e3 / min(args.steps, 100),
                   "per_step_rank0": {"p50_ms": alt["p50_ms"], "p99_ms": alt["p99_ms"], "max_ms": alt["max_ms"]},
                   "what": "the same cycle with the other inventory policy (live = a fresh NVML UUID/minor/MemoryInfo query "
                           "inside every cycle, the round-1 behaviour)"},
        "full_walk": {"value": f_units / f_kern_s, "unit": UNIT, "steps": args.full_steps,
                      "ms_per_step": f_kern_s * 1e3 / args.full_steps,
                      "e2e": {"value": f_units / f_wall_s, "unit": UNIT, "ms_per_step": f_wall_s * 1e3 / args.full_steps},
                      "window_bytes": arena,
                      "roofline": {"bound": "hbm", "achieved": f_achieved, "peak": peak, "unit": "GB/s",
                                   "frac": f_achieved / peak, "traffic": prof.get("full_walk_dram_bytes_per_launch"),
                                   "traffic_source": traffic_src, "algorithmic_bytes_per_launch": 2 * arena}},
        "clocks": clocks,
    }
    if tr:
        tl = tr["last"]
        line["transient"] = {
            "e2e_value": args.transient_steps * world / tr_wall_s, "unit": UNIT, "steps": args.transient_steps,
            "ms_per_step": tr_wall_s * 1e3 / args.transient_steps, "kernel_ms_per_step": tr["kernel_ns"] / 1e6 / args.transient_steps,
            "alloc_map_free_ms_per_step": (tr["wall_ns"] - tr["kernel_ns"]) / 1e6 / args.transient_steps,
            "roofline": {"bound": "hbm", "achieved": 2 * window * args.transient_steps / (tr["kernel_ns"] / 1e9) / 1e9, "peak": peak,
                         "unit": "GB/s", "frac": 2 * window * args.transient_steps / (tr["kernel_ns"] / 1e9) / 1e9 / peak,
                         "kernels": "probe_bulk_dyn<FILL> (W written) + probe_bulk<VERIFY> (W read), two launches",
                         "algorithmic_bytes_per_cycle": 2 * window},
            "per_step_rank0": {"p50_ms": tr["p50_ms"], "p99_ms": tr["p99_ms"], "max_ms": tr["max_ms"]},
            "bytes_walked": tl.probe.bytes_walked, "transient_flag": tl.transient,
            "what": "no standing arena (the daemon's default): per cycle cuMemCreate + map of one window, FILL, VERIFY, unmap + "
                    "release; HBM traffic 2*W like VERIFY_REFILL; between cycles the plugin holds no HBM beyond its context"}
    if node is not None:
        line["node_cycle"] = node
        if "step_ms" in node:
            node["vs_single_gpu_cycle"] = {"single_gpu_e2e_p50_ms": head["p50_ms"],
                                           "node_p50_over_single_p50": node["step_ms"]["p50"] / head["p50_ms"]}
    if line_cpu is not None:
        line["cpu_baseline"] = line_cpu
    if world == 1 and not args.no_allocate:
        try:
            line["allocate"] = bench_allocate("ours", args.quick_allocate)
            line["allocate"]["python_front_end"] = bench_allocate("ours_py", True)
        except Exception as e:  # noqa: BLE001
            line["allocate"] = {"error": str(e)}
    if args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in head["captured"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--window-gib", type=int, default=1)
    ap.add_argument("--full-steps", type=int, default=10)
    ap.add_argument("--variant", default="auto", choices=["auto", "direct", "cpasync", "bulk", "bulkw", "bulkd"])
    ap.add_argument("--cpu-iters", type=int, default=3000, help="reference cycles timed for cpu_baseline (about 10 s of CPU work)")
    ap.add_argument("--ref-cycles-per-step", type=int, default=50, help="--impl reference: node cycles per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inventory", default="snapshot", choices=["snapshot", "live"],
                    help="headline cycle's inventory policy (the other one is measured as a side leg)")
    ap.add_argument("--transient-steps", type=int, default=20)
    ap.add_argument("--no-transient", action="store_true")
    ap.add_argument("--node-steps", type=int, default=200)
    ap.add_argument("--no-node-cycle", action="store_true")
    ap.add_argument("--no-allocate", action="store_true")
    ap.add_argument("--quick-allocate", action="store_true")
    ap.add_argument("--allocate-only", action="store_true", help="host-only: print just the Allocate() leg")
    ap.add_argument("--allocate-impl", default="", choices=["", "ours", "ours_py", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the headline cycle returned in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.allocate_only):
        ap.error("--dump-outputs writes the outputs of our arm's headline cycle")
    if args.warmup < 3:
        args.warmup = 3
    if args.allocate_only:
        print(json.dumps(bench_allocate(args.allocate_impl or ("reference" if args.impl == "reference" else "ours"),
                                        args.quick_allocate)))
        return
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_ours(args)
    if int(os.environ.get("WORLD_SIZE", 1)) > 1:
        import torch.distributed as dist
        if dist.is_initialized():
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
