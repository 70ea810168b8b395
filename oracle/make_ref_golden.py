"""Records what oracle/_ref/ref_inventory answers into tests/golden/, so that the tests compare against the reference
without needing its sources. ref_inventory is the C restatement of the reference's NVML path, and `make -C oracle` links
it with the reference's own nvml_dl.c. TEST INFRASTRUCTURE.

Run from the repo root, after `make -C oracle` has built oracle/_ref/:
    python oracle/make_ref_golden.py          8 synthetic B200s of oracle/_fake -> tests/golden/ref_inventory_fake.json
    python oracle/make_ref_golden.py --b200   the real NVML of a B200 box       -> tests/golden/ref_inventory_b200.json

Each run keeps the command line, the variables it adds to the environment (null: no NVML on the library path at all),
the exit code, stdout and stderr. Where the binary wrote the ListAndWatchResponse (`--lw-out`, the file name left out)
the SHA-256 of those bytes is kept. Timings inside stdout are whatever the recording machine measured.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "ref_inventory")
FAKE = os.path.join(ROOT, "oracle", "_fake")

FAKE_RUNS = [
    (["inventory"], None),
    *[(["inventory", "--lw-out"], {"FAKE_NVML_GPUS": str(n)}) for n in (1, 2, 8)],
    (["inventory", "--unit", "MiB"], {"FAKE_NVML_GPUS": "1"}),
    (["bench", "--iters", "2"], {"FAKE_NVML_GPUS": "8"}),
    *[(["bench", "--iters", "3", "--warmup", "1", "--gpus", str(n)], {"FAKE_NVML_GPUS": "8"}) for n in (1, 2, 4)],
    (["inventory", "--gpus", "2"], {"FAKE_NVML_GPUS": "8"}),
]
B200_RUNS = [(["inventory", "--unit", "GiB", "--lw-out"], {}), (["inventory", "--unit", "MiB"], {})]


def record(args, env, lib_dir):
    e = dict(os.environ)
    if env is None:
        e.pop("LD_LIBRARY_PATH", None)
    else:
        if lib_dir:
            e["LD_LIBRARY_PATH"] = lib_dir
        e.update(env)
    with tempfile.TemporaryDirectory() as d:
        lw = os.path.join(d, "lw.bin")
        argv = [REF_BIN] + args + ([lw] if args[-1] == "--lw-out" else [])
        out = subprocess.run(argv, env=e, capture_output=True, text=True, timeout=300)
        r = {"args": args, "env": env, "returncode": out.returncode, "stdout": out.stdout, "stderr": out.stderr}
        if args[-1] == "--lw-out" and out.returncode == 0:
            with open(lw, "rb") as f:
                r["lw_sha256"] = hashlib.sha256(f.read()).hexdigest()
    return r


def main():
    if not os.access(REF_BIN, os.X_OK):
        sys.exit(f"{REF_BIN} is not built: make -C oracle REF=<reference checkout>")
    b200 = "--b200" in sys.argv[1:]
    runs = [record(a, e, None if b200 else FAKE) for a, e in (B200_RUNS if b200 else FAKE_RUNS)]
    name = "ref_inventory_b200.json" if b200 else "ref_inventory_fake.json"
    out = {"_comment": "recorded by oracle/make_ref_golden.py" + (" --b200" if b200 else "") + " from oracle/_ref/ref_inventory",
           "runs": runs}
    with open(os.path.join(ROOT, "tests", "golden", name), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
