"""The routing contract of the C entry points: for every kernel-path override, family knob set, entry point, geometry,
padding, mode and element type, the status, the kernel family that ran (ts_last_kernel_path), the number of kernels
launched and the backward workspace size must equal tests/golden/dispatch_table.json.xz (tests/golden/make_dispatch_table.py
recorded it and runs the same cases here)."""
import importlib.util
from pathlib import Path

import pytest
import torch

GOLDEN = Path(__file__).resolve().parent / "golden"

pytestmark = pytest.mark.gpu


def _generator():
    spec = importlib.util.spec_from_file_location("make_dispatch_table", GOLDEN / "make_dispatch_table.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.fixture()
def default_steering():
    from torchshifts.extension import native
    lib = native().lib
    knobs = b"use_tma=1,use_halo=1,use_flat=1"
    lib.ts_set_kernel_path(0)
    lib.ts_set_tuning(knobs)
    yield
    lib.ts_set_kernel_path(0)
    lib.ts_set_tuning(knobs)


def test_dispatch_table_matches_recording(default_steering):
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    gen = _generator()
    recorded = gen.load()
    table = gen.run_table()
    assert (table["forced"], table["knobs"]) == (recorded["forced"], recorded["knobs"])
    steerings = [f"forced={f},{k}" for f in recorded["forced"] for k in recorded["knobs"]]
    for section in ("workspace", "cases"):
        assert list(table[section]) == list(recorded[section]), f"{section}: the case list differs from the recording"
        bad = []
        for key, want in recorded[section].items():
            got = table[section][key]
            if got == want:
                continue
            if section == "cases":      # three digits per steering: status, last kernel path, launches
                got, want = ([c[i:i + 3] for i in range(0, len(c), 3)] for c in (got, want))
                bad += [f"{key} {s}: status/path/launches {g} != {w}" for s, g, w in zip(steerings, got, want) if g != w]
            else:
                bad.append(f"{key}: workspace bytes {got} != {want}")
        assert not bad, f"{len(bad)} {section} mismatches, first: " + "; ".join(bad[:20])
