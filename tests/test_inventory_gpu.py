"""GPU-box parity of the inventory half against the reference's own NVML path. The C restatement linked with the
reference's nvml_dl.c (oracle/_ref/ref_inventory) was run on a B200, and its answer is recorded in
tests/golden/ref_inventory_b200.json. Every field the plugin consumes must agree with it bit for bit: total bytes,
MiB, slice count, and the ListAndWatchResponse bytes. The card's identity (uuid, minor, bus id, device order)
differs from card to card, so it is checked against NVML on this box through pynvml, an independent binding of
the same libnvidia-ml calls the reference makes, and the recorded card's uuid is exchanged for this card's."""
import hashlib
import json
import re

import pytest

from oracle import wire_oracle as wo
from tests.ref_answers import recorded

pytestmark = pytest.mark.gpu


def run_ref(unit="GiB"):
    args = ["inventory", "--unit", unit] + (["--lw-out"] if unit == "GiB" else [])
    out = recorded("ref_inventory_b200.json", args, {})
    return json.loads(out.stdout), getattr(out, "lw_sha256", None)


def nvml_identity():
    import pynvml as nv
    nv.nvmlInit()
    s = lambda x: x.decode() if isinstance(x, bytes) else x  # noqa: E731
    hs = [nv.nvmlDeviceGetHandleByIndex(i) for i in range(nv.nvmlDeviceGetCount())]
    return [{"uuid": s(nv.nvmlDeviceGetUUID(h)), "minor": nv.nvmlDeviceGetMinorNumber(h),
             "bus_id": s(nv.nvmlDeviceGetPciInfo(h).busId)} for h in hs]


def test_recorded_reference_answer_comes_from_a_b200():
    for unit in ("GiB", "MiB"):
        ref, _ = run_ref(unit)
        assert ref["mode"] == "inventory" and ref["unit"] == unit and ref["n_gpus"] == len(ref["devices"]) >= 1
        assert all(d["model"] == "NVIDIA B200" for d in ref["devices"])


def test_inventory_matches_reference_nvml_path(gsb):
    ref, ref_lw_sha = run_ref()
    theirs = ref["devices"][0]
    n = gsb.device_count()
    infos = [gsb.device_info(i) for i in range(n)]
    ident = nvml_identity()
    assert n == len(ident) >= 1
    for mine, nv in zip(infos, ident):
        assert mine.uuid == nv["uuid"] and re.fullmatch(r"GPU-[0-9a-f]{8}(-[0-9a-f]{4}){3}-[0-9a-f]{12}", mine.uuid)
        assert mine.minor == nv["minor"]
        assert mine.bus_id.lower() == nv["bus_id"].lower() and len(mine.bus_id) == len(theirs["bus_id"])
        assert mine.total_bytes == theirs["total_bytes"]
        assert mine.total_mib == theirs["memory_mib"]
        assert mine.cc == (10, 0) and mine.sm_count == 148
    # the reference derives the process-global slice count from device 0 only (nvidia.go:70-72)
    s = gsb.slices(infos[0].total_mib, True)
    assert s == ref["gpu_memory"] == infos[0].total_bytes >> 30
    lw = gsb.encode_list_and_watch([i.uuid for i in infos], s)
    # one GPU's list is the reference's bytes with the recorded card's uuid in place of this one's; a node's list is
    # the GPUs' lists one after another (a repeated field), in device order
    per_gpu = [gsb.encode_list_and_watch([i.uuid], s) for i in infos]
    assert lw == b"".join(per_gpu)
    for i, one in zip(infos, per_gpu):
        assert hashlib.sha256(one.replace(i.uuid.encode(), theirs["uuid"].encode())).hexdigest() == ref_lw_sha
        assert len(one) == ref["lw_len"]
    # ... and both equal the pure-Python restatement of getDevices + gogo marshal
    devs, _, mem = wo.getDevices([{"uuid": d["uuid"], "path": d["path"], "memory_mib": d["memory_mib"]}
                                  for d in ref["devices"]])
    assert mem == s and hashlib.sha256(wo.marshal_ListAndWatchResponse(devs)).hexdigest() == ref_lw_sha
    devs, name_map, mem = wo.getDevices([{"uuid": i.uuid, "path": f"/dev/nvidia{i.minor}", "memory_mib": i.total_mib}
                                         for i in infos])
    assert mem == s and wo.marshal_ListAndWatchResponse(devs) == lw
    assert name_map == {i.uuid: i.minor for i in infos}
    assert gsb.fake_device_id(infos[0].uuid, 0) == ref["first_id"].replace(theirs["uuid"], infos[0].uuid)
    assert gsb.fake_device_id(infos[-1].uuid, s - 1) == ref["last_id"].replace(ref["devices"][-1]["uuid"], infos[-1].uuid)


def test_b200_advertises_179_slices(gsb):
    info = gsb.device_info(0)
    # nvidia-smi's 183359 MiB; cuDeviceTotalMem alone would give 178 (profiles/envprobe_r01.txt)
    assert info.total_mib == 183359 and gsb.slices(info.total_mib, True) == 179
    assert info.cuda_total_bytes >> 30 == 178
    assert len(gsb.encode_list_and_watch([info.uuid], 179)) == 10451  # SURVEY.md §8(a) a7


def test_mib_unit_matches_reference(gsb):
    ref, _ = run_ref("MiB")
    info = gsb.device_info(0)
    assert gsb.slices(info.total_mib, False) == ref["gpu_memory"] == 183359
