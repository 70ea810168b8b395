"""The reference's recorded answers: what oracle/_ref/ref_inventory printed for a command line, as
oracle/make_ref_golden.py stored it under tests/golden/. ref_inventory is the C restatement of the reference's NVML
path, linked with the reference's own nvml_dl.c. The tests compare against these answers instead of running the
binary, which can only be built where the reference's sources are."""
import json
import os
from types import SimpleNamespace

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def recorded(fixture: str, args, env=None) -> SimpleNamespace:
    """The run of `ref_inventory <args>` recorded in tests/golden/<fixture>, with the variables `env` added to the
    environment (None: no NVML on the library path at all). `--lw-out` stands without its file name; such a run
    carries lw_sha256, the SHA-256 of the ListAndWatchResponse bytes it wrote."""
    with open(os.path.join(GOLDEN, fixture)) as f:
        runs = json.load(f)["runs"]
    for r in runs:
        if r["args"] == list(args) and r["env"] == env:
            return SimpleNamespace(**r)
    raise KeyError(f"{fixture} has no run of ref_inventory {' '.join(args)} with {env}: record it with "
                   "oracle/make_ref_golden.py")
