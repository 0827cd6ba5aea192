"""The persistent kernel families (TMA, staged, halo, flat) in every planner regime, whole tensors against the oracle.

The planners (plan_tma, plan_staged, plan_halo, plan_flat, plan_units, pick_unit_images) decide which branch of the
tile, stage, unit and ring code a call runs.  At the small shapes of the sweep tests they take almost only one branch:
one tile per plane, one unit per CTA, a ring that barely wraps.  Each case below forces one family
(ts_set_kernel_path), sets tuning knobs (ts_set_tuning) and picks a geometry that drives the planner into a named
regime.  Before it runs, the case reads the plan through ts_debug_route and asserts the family and every regime it
claims, so a case that drifts out of its regime fails instead of passing without testing anything.  It then runs
through the public functional API and autograd and compares WHOLE tensors with the oracle:

* fp32, fp64, integer: forward and grad_input bit-exact;
* 16-bit: equal to the fp32 oracle rounded once to the storage type (mixed precision: the oracle gets the unrounded
  fp32 weights; same-dtype layers: the 16-bit weights);
* grad_weight: rtol 1e-5 against the fp64 oracle, atol 1e-5 * max|gw| (a 16-bit grad_weight: plus half an ulp of its
  type, the one rounding of its store).

Knob invariance (test_knobs_leave_results_bit_identical) is checked bit for bit; the comment above it gives the two
cases where the code itself regroups the grad_weight sums.

Weights are chosen per channel: every residue of the last-axis shift modulo the 16-byte item width, ties at +-k.5,
-0.0, fractions just below 1, shifts past a tile and past the plane (_weights).

The CPU-side test pins ts_debug_route's argument checks; everything else needs a B200.
"""
import ctypes as ct
from dataclasses import dataclass, field

import numpy as np
import pytest
import torch

from oracle.oracle import check_borders, quantize_shift_weights_np, split_backward, split_forward

GENERIC, STAGED, TMA, HALO, FLAT = 1, 2, 3, 5, 6
TS_OK, TS_ERR_INVALID_ARGUMENT, TS_ERR_NO_DEVICE = 0, 1, 7
TS_WEIGHTS_F32 = 0x100
N_OUT = 13
# ts_debug_route's fields after out[0] (the path)
FIELDS = ("tiles", "tiles_a", "tiles_b", "tiles_g", "np", "npu", "units", "grid", "stages", "warps", "slots", "table")
# the defaults of tuning() in ts_capi.cu: every knob the cases set goes back to these
DEFAULT_TUNING = (b"stages=0,stage_kb=0,warps=15,ctas_per_sm=1,chunk_planes=0,tma_stages=0,tma_warps=0,use_tma=1,"
                  b"tma_stage_kb=0,nhwc_variant=0,nhwc_ring_rows=0,nhwc_rows_warps=0,use_halo=1,halo=0,halo_stages=0,"
                  b"halo_warps=0,unit_order=1,use_flat=1,flat_ctas=0,flat_stage_kb=0,flat_stages=0,flat_warps=0,"
                  b"cl_ahead=0,cl_rows=0")
FIXCAP = 1536          # ts_halo.cu: cells of one fixer list; a unit that needs more is patched without a list
DTYPES = {  # name -> (storage dtype, weight dtype, ts dtype code, element bytes)
    "f32": (torch.float32, torch.float32, 0, 4), "f64": (torch.float64, torch.float64, 1, 8),
    "f16": (torch.float16, torch.float16, 2, 2), "bf16": (torch.bfloat16, torch.bfloat16, 3, 2),
    "f16m": (torch.float16, torch.float32, 2 | TS_WEIGHTS_F32, 2), "bf16m": (torch.bfloat16, torch.float32, 3 | TS_WEIGHTS_F32, 2),
    "q1": (torch.quint8, None, -1, 1), "q4": (torch.qint32, None, -1, 4),
}


@dataclass
class Case:
    name: str
    path: int                 # forced family of the phases in `ops`
    kind: str                 # "sparse", "active" or "quant"
    dtype: str
    shape: tuple
    pads: tuple = (0,)
    crops: tuple = (None,)    # each: None or [dim][2] (left_cut, right_cut)
    knobs: str = ""
    ops: tuple = ("fwd", "bwd")   # phases run on the forced family; the others run under automatic routing
    claims: tuple = ()
    fused: bool = False       # backward through FusedGradWeightAllReduce (one rank)
    weights: dict = field(default_factory=dict)   # channel -> explicit weights row

    @property
    def dim(self):
        return len(self.shape) - 2


CASES = [
    # ---------------------------------------------------------------- TMA
    Case("tma_2d_f32_gather_tiles", TMA, "sparse", "f32", (3, 160, 40, 260), crops=([[1, 2], [0, 0]],),
         knobs="tma_stage_kb=8,tma_stages=2,chunk_planes=1", ops=("fwd",),
         claims=("tma.gather.4B", "tma.col_tiles.4B", "tma.row_tiles", "tma.units_gt_grid", "tma.stages2",
                 "tma.shift.row", "tma.shift.col")),
    Case("tma_2d_f32_sparse_tiles", TMA, "sparse", "f32", (2, 100, 37, 260), knobs="tma_stage_kb=16,unit_order=0,chunk_planes=1",
         claims=("tma.bwd_sparse.2d", "tma.row_tiles", "tma.col_tiles.4B", "tma.unit_order0", "tma.units_gt_grid")),
    Case("tma_2d_f32_active_tiles", TMA, "active", "f32", (2, 100, 37, 260), knobs="tma_stage_kb=16,unit_order=0,chunk_planes=1",
         claims=("tma.active_fwd.2d", "tma.bwd_active.2d", "tma.row_tiles", "tma.col_tiles.4B", "tma.unit_order0")),
    Case("tma_3d_f32_sparse", TMA, "sparse", "f32", (2, 12, 19, 12, 32), knobs="tma_stage_kb=16,tma_warps=1",
         claims=("tma.bwd_sparse.3d", "tma.slab_tiles", "tma.warps1", "tma.shift.slab")),
    Case("tma_3d_f32_active", TMA, "active", "f32", (2, 12, 19, 12, 32), knobs="tma_stage_kb=16",
         claims=("tma.active_fwd.3d", "tma.bwd_active.3d", "tma.slab_tiles", "tma.shift.slab")),
    Case("tma_1d_f32_sparse", TMA, "sparse", "f32", (16, 40, 1000), knobs="chunk_planes=1,tma_warps=31",
         claims=("tma.bwd_sparse.1d", "tma.col_tiles.4B", "tma.warps_max", "tma.units_gt_grid", "pass2.many_slots",
                 "tma.shift.col")),
    Case("tma_1d_f32_active_fused", TMA, "active", "f32", (16, 40, 1000), knobs="chunk_planes=1,tma_warps=31", fused=True,
         claims=("tma.active_fwd.1d", "tma.bwd_active.1d", "tma.warps_max", "pass2.many_slots", "pass2.fused")),
    Case("tma_2d_f32_ragged_stage", TMA, "active", "f32", (37, 12, 8, 32), knobs="chunk_planes=30",
         claims=("tma.np_ragged", "tma.units_ragged")),
    Case("tma_2d_u8_ragged_stage", TMA, "quant", "q1", (50, 40, 8, 64), crops=(None, [[1, 0], [0, 16]]),
         claims=("tma.gather.1B", "tma.np_ragged")),
    Case("tma_2d_f64_ragged_stage", TMA, "sparse", "f64", (30, 8, 8, 32), ops=("fwd",), claims=("tma.gather.8B", "tma.np_ragged")),
    Case("tma_2d_f16_gather_cols", TMA, "sparse", "f16", (3, 24, 10, 264), ops=("fwd",), claims=("tma.gather.2B", "tma.col_tiles.2B")),
    Case("tma_2d_bf16m_sparse", TMA, "sparse", "bf16m", (3, 24, 12, 264), knobs="tma_warps=31",
         claims=("tma.mixed16.gather", "tma.mixed16.bwd_sparse", "tma.col_tiles.2B", "tma.warps_max")),
    Case("tma_2d_f16m_active", TMA, "active", "f16m", (3, 24, 13, 264), knobs="tma_stage_kb=2,tma_stages=2",
         claims=("tma.mixed16.active_fwd", "tma.mixed16.bwd_active", "tma.col_tiles.2B", "tma.row_tiles", "tma.stages2")),
    # ---------------------------------------------------------------- staged
    Case("staged_3d_sparse_slabs", STAGED, "sparse", "f32", (5, 12, 13, 8, 16), pads=(0, 1, 2, 3, 4),
         crops=(None, [[1, 1], [1, 0], [0, 4]]), knobs="stage_kb=3,stages=8",
         claims=("staged.slab_tiles", "staged.stages8") + tuple(f"staged.pad{p}{c}" for p in range(5) for c in ("", ".crop"))),
    Case("staged_3d_active_slabs", STAGED, "active", "f32", (5, 12, 13, 8, 16), pads=(0, 1, 2, 3, 4),
         crops=(None, [[1, 1], [1, 0], [0, 4]]), knobs="stage_kb=3,warps=1", claims=("staged.slab_tiles", "staged.warps1")),
    Case("staged_2d_gather_vec8", STAGED, "sparse", "f32", (20, 40, 4, 10), pads=(0, 2, 3), ops=("fwd",),
         knobs="stage_kb=1,ctas_per_sm=2,stages=2,chunk_planes=9",
         claims=("staged.vec8", "staged.np_ragged", "staged.units_ragged", "staged.ctas_per_sm", "staged.stages2")),
    Case("staged_2d_gather_vec4", STAGED, "sparse", "f32", (20, 64, 4, 9), pads=(1, 4), ops=("fwd",),
         knobs="stage_kb=1,warps=31,unit_order=0", claims=("staged.vec4", "staged.np_ragged", "staged.warps31", "staged.unit_order0")),
    Case("staged_2d_gather_u8", STAGED, "quant", "q1", (20, 48, 4, 20), pads=(0, 3), crops=(None, [[1, 0], [0, 0]]),
         knobs="warps=1", claims=("staged.vec4",)),
    Case("staged_2d_gather_vec16", STAGED, "sparse", "f32", (6, 16, 8, 32), pads=(0, 4), ops=("fwd",), claims=("staged.vec16",)),
    Case("staged_2d_bf16", STAGED, "active", "bf16", (6, 24, 10, 16), pads=(0, 3), crops=(None, [[1, 2], [0, 8]]),
         claims=("staged.half.bf16",)),
    Case("staged_2d_f16", STAGED, "sparse", "f16", (6, 24, 10, 16), pads=(1, 4), crops=(None, [[0, 1], [8, 0]]),
         knobs="unit_order=0,chunk_planes=1", claims=("staged.half.f16",)),
    Case("staged_2d_unit_order0_bwd", STAGED, "active", "f32", (2, 160, 6, 16), pads=(2,), knobs="unit_order=0",
         claims=("staged.unit_order0",)),
    # ---------------------------------------------------------------- halo
    Case("halo_2d_active", HALO, "active", "f32", (13, 40, 20, 24), pads=(0, 1, 2, 3, 4), crops=(None, [[1, 0], [4, 4]]),
         knobs="halo_stages=2",
         claims=("halo.classes_all5", "halo.beyond", "halo.np_ragged", "halo.stages2", "halo.2d", "halo.crop")
         + tuple(f"halo.pad{p}" for p in range(5))),
    Case("halo_2d_sparse_bwd", HALO, "sparse", "f32", (3, 160, 20, 24), pads=(1, 3), crops=(None, [[2, 1], [0, 4]]),
         knobs="unit_order=0,chunk_planes=1", ops=("bwd",), claims=("halo.unit_order0", "halo.classes_all5", "halo.crop")),
    Case("halo_2d_halo1", HALO, "active", "f32", (4, 16, 12, 16), pads=(2, 4), knobs="halo=1", claims=("halo.beyond",)),
    Case("halo_3d", HALO, "active", "f32", (3, 8, 6, 10, 16), pads=(0, 1, 2, 3, 4), crops=(None, [[1, 0], [0, 2], [0, 4]]),
         claims=("halo.3d", "halo.crop") + tuple(f"halo.pad{p}" for p in range(5))),
    Case("halo_3d_sparse_bwd", HALO, "sparse", "f32", (3, 8, 6, 10, 16), pads=(0, 3), ops=("bwd",), claims=("halo.3d",)),
    Case("halo_2d_no_table", HALO, "active", "f32", (2, 600, 8, 16), pads=(2,), claims=("halo.no_table",)),
    Case("halo_2d_fix_without_list", HALO, "active", "f32", (2, 4, 64, 64), pads=(3, 1), knobs="halo=16",
         weights={0: [16.25, 16.5], 1: [-15.75, 15.0], 2: [12.5, -15.5]}, claims=("halo.fixcap",)),
    # ---------------------------------------------------------------- flat
    Case("flat_2d_f32", FLAT, "sparse", "f32", (7, 13, 6, 12), ops=("fwd",), knobs="flat_stage_kb=1,flat_stages=2,flat_warps=1",
         claims=("flat.f32", "flat.np_ragged", "flat.stages2", "flat.warps1")),
    Case("flat_2d_u8", FLAT, "quant", "q1", (20, 40, 8, 24), knobs="flat_ctas=2,flat_stage_kb=1", claims=("flat.q1", "flat.ctas")),
    Case("flat_2d_q32_no_table", FLAT, "quant", "q4", (3, 600, 4, 8), claims=("flat.q4", "flat.no_table", "flat.np_ragged")),
    Case("flat_1d_f32", FLAT, "sparse", "f32", (8, 12, 100), ops=("fwd",), claims=("flat.f32",)),
]

REQUIRED = (
    ["tma.col_tiles.4B", "tma.col_tiles.2B", "tma.row_tiles", "tma.slab_tiles", "tma.np_ragged", "tma.units_ragged",
     "tma.units_gt_grid", "tma.stages2", "tma.unit_order0", "tma.warps1", "tma.warps_max",
     "tma.shift.row", "tma.shift.col", "tma.shift.slab",
     "tma.gather.1B", "tma.gather.2B", "tma.gather.4B", "tma.gather.8B",
     "tma.mixed16.gather", "tma.mixed16.active_fwd", "tma.mixed16.bwd_sparse", "tma.mixed16.bwd_active"]
    + [f"tma.{k}.{d}d" for k in ("active_fwd", "bwd_sparse", "bwd_active") for d in (1, 2, 3)]
    + ["staged.slab_tiles", "staged.vec16", "staged.vec8", "staged.vec4", "staged.np_ragged", "staged.units_ragged",
       "staged.unit_order0", "staged.stages2", "staged.stages8", "staged.warps1", "staged.warps31", "staged.ctas_per_sm",
       "staged.half.f16", "staged.half.bf16"]
    + [f"staged.pad{p}{c}" for p in range(5) for c in ("", ".crop")]
    + ["halo.classes_all5", "halo.beyond", "halo.fixcap", "halo.no_table", "halo.stages2", "halo.np_ragged",
       "halo.unit_order0", "halo.2d", "halo.3d", "halo.crop"] + [f"halo.pad{p}" for p in range(5)]
    + ["flat.np_ragged", "flat.ctas", "flat.stages2", "flat.warps1", "flat.no_table", "flat.q1", "flat.q4", "flat.f32"]
    + ["pass2.many_slots", "pass2.fused"])


# ------------------------------------------------------------------------------------------ fixtures and helpers
@pytest.fixture(scope="module")
def lib():
    from torchshifts.extension import native
    return native().lib


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


def _restore(lib):
    lib.ts_set_kernel_path(0)
    assert lib.ts_set_tuning(DEFAULT_TUNING) == TS_OK


@pytest.fixture(scope="module")
def steering(lib):
    """Sets (path, knobs); the forced path and every knob go back to tuning()'s defaults after each use and after the
    module, also when a test fails."""
    class Steer:
        def __call__(self, path, knobs=""):
            _restore(lib)
            assert lib.ts_set_tuning(knobs.encode()) == TS_OK, knobs
            lib.ts_set_kernel_path(path)

    _restore(lib)
    try:
        yield Steer()
    finally:
        _restore(lib)


@pytest.fixture()
def steer(steering, lib):
    try:
        yield steering
    finally:
        _restore(lib)


def _item(case):
    """Elements per 16-byte item of the last axis (4: the halo family's word misalignment classes)."""
    return 4 if case.path == HALO else 16 // DTYPES[case.dtype][3]


def _weights(case, rng):
    """[C, dim] fp32.  Channel c, category c % 10: large shifts first (3/4 of the axis: past a tile whenever the axis has
    two or more; the axis + 3 or + 5: past the plane), then fractions: 0.5 ties, 1 - 2^-18 (just below 1), exact
    integers, random; channel 1 is -0.0 on every axis.  The last axis' integer part is (c mod item) - item / 2 plus the
    large shift rounded outwards to a whole number of items, so the channels run through every residue modulo the item
    width."""
    C, dim, sizes = case.shape[1], case.dim, case.shape[2:]
    item = _item(case)
    w = np.zeros((C, dim), dtype=np.float64)
    for c in range(C):
        cat = c % 10
        for a in range(dim):
            S = sizes[a]
            base = (c % item) - item // 2 if a == dim - 1 else int(rng.integers(-3, 4))
            big = (3 * S // 4, 0, S + 3, 0, -(3 * S // 4), -(S + 5), 0, 0, 0, 0)[cat]
            if a == dim - 1 and big:
                big = -(-big // item) * item if big > 0 else (big // item) * item
            frac = (0.25, 0.0, 0.5, 1.0 - 2.0 ** -18, 0.75, 0.5, 0.5, rng.uniform(0.05, 0.45), 0.0,
                    rng.uniform(0.05, 0.95))[cat]
            w[c, a] = base + big + frac
    w[1 % C, :] = -0.0
    for c, row in case.weights.items():
        w[c, :] = row
    return w.astype(np.float32)


def _geometry(case, crop):
    from torchshifts._cabi import make_geometry
    lb, rb = check_borders(case.dim, case.shape[2:], crop)
    strides, s = [], 1
    for v in reversed(case.shape):
        strides.insert(0, s)
        s *= v
    return make_geometry(case.dim, case.shape, strides, lb, rb), lb, rb


def _route(lib, case, pad, crop, op):
    geo, _, _ = _geometry(case, crop)
    out = (ct.c_int64 * N_OUT)()
    code, es = DTYPES[case.dtype][2], DTYPES[case.dtype][3]
    rc = lib.ts_debug_route(ct.byref(geo), op, code, es, pad, 1 if case.kind == "active" else 0, out, N_OUT)
    assert rc == TS_OK, (case.name, pad, crop, op, rc)
    r = dict(zip(FIELDS, list(out)[1:]))
    r["path"] = out[0]
    return r


def _phases(case):
    fwd_op = 1 if case.kind == "active" else 0
    return [(p, fwd_op if p == "fwd" else 2) for p in case.ops if not (p == "bwd" and case.kind == "quant")]


def _reduce_shift(s, n, pad):
    """ts_common.cuh reduce_shift (C remainder: the sign of s)."""
    if n <= 1:
        return 0
    period = {2: n, 3: 2 * (n - 1), 4: 2 * n}.get(pad, 0)
    if period == 0:
        return int(max(-(n + 1), min(n + 1, s)))
    return int(np.fmod(s, period))


def _halo_units(case, w, pad, crop, mode):
    """Host mirror of ts_halo.cu compute_unit_shift / unit_geom / classify and of the fixer's HaloRange cell count:
    -> per channel (class 0..4, fits, x cells, grad cells)."""
    hr = int(dict(kv.split("=") for kv in case.knobs.split(",") if kv).get("halo", 0)) or 4
    hc = (hr + 3) // 4 * 4
    d = case.dim
    _, lb, rb = _geometry(case, crop)
    S, OS = case.shape[2:], [rb[a] - lb[a] for a in range(d)]
    B, L, OB, OL, lbB, lbL = S[d - 2], S[d - 1], OS[d - 2], OS[d - 1], lb[d - 2], lb[d - 1]
    px, bpx, pg, bpg = L + 2 * hc, B + 2 * hr, OL + 2 * hc, OB + 2 * hr
    px += 4 if px % 8 == 0 else 0
    pg += 4 if pg % 8 == 0 else 0
    bwd, active = mode == 2, case.kind == "active"
    IB, IG = (B, L // 4) if bwd else (OB, OL // 4)

    def cells(lo_r, hi_r, lo_c, hi_c, rows, cols):
        nr = (-lo_r if lo_r < 0 else 0) + (hi_r - (rows - 1) if hi_r > rows - 1 else 0)
        nc = (-lo_c if lo_c < 0 else 0) + (hi_c - (cols - 1) if hi_c > cols - 1 else 0)
        return nr * (hi_c - lo_c + 1) + rows * nc

    iw, _ = split_backward(w, active) if bwd else split_forward(w, active)
    units = []
    for c in range(w.shape[0]):
        sx = [_reduce_shift(int(iw[c, a]), S[a], pad) for a in (d - 2, d - 1)]
        sg = [_reduce_shift(int(iw[c, a]), OS[a], pad) for a in (d - 2, d - 1)]
        xr0, xc0 = (0 if bwd else lbB) - sx[0] + hr, (0 if bwd else lbL) - sx[1] + hc
        fits = xr0 >= 0 and xr0 + IB <= bpx - 1 and xc0 >= 0 and xc0 + 4 * IG <= px - 1
        ex = 1 if active else 0
        sgr, sgc = (-sg[0], -sg[1]) if active else (sg[0], sg[1])
        gc0, vc0 = -lbL + sgc + hc, -lbL + (0 if d == 3 else hc)
        if bwd:
            fits = fits and sgr + hr >= 0 and OB - 1 + sgr + hr + ex <= bpg - 1 and sgc + hc >= 0 and OL - 1 + sgc + hc + ex <= pg - 1
        cls = xc0 & 3 if fits else 4
        if fits and bwd and not ((vc0 & 3) == 0 and (gc0 & 3) == (xc0 & 3 if active else (4 - (xc0 & 3)) & 3)):
            cls = 4
        xlo_r, xlo_c = xr0 - hr, xc0 - hc
        nx = cells(xlo_r, xlo_r + IB, xlo_c, xlo_c + 4 * IG, B, L)
        ng = cells(sgr, OB - 1 + sgr + ex, sgc, OL - 1 + sgc + ex, OB, OL) if bwd else 0
        units.append((cls, fits, nx, ng, px * bpx < 65536 and pg * bpg < 65536))
    return units


def _knob(case, key):
    kv = dict(k.split("=") for k in case.knobs.split(",") if k)
    return int(kv[key]) if key in kv else None


def _regimes(case, pad, crop, phase, op, r, w, sms):
    """The regimes one phase of a case reaches, from its plan (ts_debug_route), its geometry and its weights."""
    reached = set()
    d, N, C = case.dim, case.shape[0], case.shape[1]
    _, lb, rb = _geometry(case, crop)
    S, OS = case.shape[2:], [rb[a] - lb[a] for a in range(d)]
    es = DTYPES[case.dtype][3]
    lev = {0: d - 3, 1: d - 2, 2: d - 1}            # level -> tensor axis (negative: absent)
    O = {k: (OS[a] if a >= 0 else 1) for k, a in lev.items()}
    fam = {TMA: "tma", STAGED: "staged", HALO: "halo", FLAT: "flat"}.get(r["path"])
    if fam is None:
        return reached
    if r["np"] > 1 and (N * C if fam == "flat" else N) % r["np"] != 0:
        reached.add(f"{fam}.np_ragged")
    if fam != "flat":
        if N % r["npu"] != 0 and (_knob(case, "chunk_planes") or 0) > 0:
            reached.add(f"{fam}.units_ragged")
        if r["units"] > r["grid"]:
            reached.add(f"{fam}.units_gt_grid")
            if _knob(case, "unit_order") == 0:
                reached.add(f"{fam}.unit_order0")
    if fam == "tma":
        ogr = O[2] * (es if op == 0 else 4 if case.dtype == "f32" else 2) // 16
        if r["tiles_g"] > 1 and ogr % r["tiles_g"] != 0:
            reached.add(f"tma.col_tiles.{es}B")
        if d >= 2 and r["tiles_b"] > 1 and O[1] % r["tiles_b"] != 0:
            reached.add("tma.row_tiles")
        if d == 3 and r["tiles_a"] > 1 and O[0] % r["tiles_a"] != 0:
            reached.add("tma.slab_tiles")
        fills = -(-r["units"] // r["grid"]) * -(-r["npu"] // r["np"]) * r["tiles"]
        if r["stages"] == 2 and _knob(case, "tma_stages") == 2 and fills >= 8:
            reached.add("tma.stages2")
        if r["warps"] == 1:
            reached.add("tma.warps1")
        if r["warps"] == (31 if op == 0 else 15):
            reached.add("tma.warps_max")
        for k, name, tiles in ((0, "slab", r["tiles_a"]), (1, "row", r["tiles_b"]), (2, "col", r["tiles_g"])):
            a = lev[k]
            if a < 0 or tiles < 2:
                continue
            mag = np.abs(w[:, a])
            if ((mag > O[k] / tiles + 1) & (mag < S[a] - 1)).any() and (mag > S[a] + 1).any():
                reached.add(f"tma.shift.{name}")
        mixed = case.dtype in ("f16m", "bf16m")
        if op == 0:
            reached.add("tma.mixed16.gather" if mixed else f"tma.gather.{es}B")
        else:
            k = "active_fwd" if op == 1 else "bwd_active" if case.kind == "active" else "bwd_sparse"
            reached.add(f"tma.mixed16.{k}" if mixed else f"tma.{k}.{d}d")
    elif fam == "staged":
        IA = S[0] if op == 2 else OS[0]
        if d == 3 and r["tiles"] > 1 and IA % r["tiles"] != 0:
            reached.add("staged.slab_tiles")
        if op == 0:
            lb_, olb = S[d - 1] * es, OS[d - 1] * es
            vb = next((v for v in (16, 8, 4) if v >= es and lb_ % v == 0 and olb % v == 0), 0)
            reached.add(f"staged.vec{vb}")
            if (_knob(case, "ctas_per_sm") or 1) > 1 and r["grid"] > sms:
                reached.add("staged.ctas_per_sm")
            if r["warps"] == 31:
                reached.add("staged.warps31")
        for k in (2, 8):
            if r["stages"] == k and _knob(case, "stages") == k:
                reached.add(f"staged.stages{k}")
        if r["warps"] == 1:
            reached.add("staged.warps1")
        if case.dtype in ("f16", "bf16"):
            reached.add(f"staged.half.{case.dtype}")
        reached.add(f"staged.pad{pad}" + (".crop" if crop is not None else ""))
    elif fam == "halo":
        units = _halo_units(case, w, pad, crop, op)
        classes = {u[0] for u in units}
        if classes == {0, 1, 2, 3, 4}:
            reached.add("halo.classes_all5")
        if any(not u[1] for u in units):
            reached.add("halo.beyond")
        if pad != 0 and any(u[1] and u[4] and max(u[2], u[3]) > FIXCAP for u in units):
            reached.add("halo.fixcap")
        if r["table"] == 0 and C > 512:
            reached.add("halo.no_table")
        if r["stages"] == 2 and _knob(case, "halo_stages") == 2:
            reached.add("halo.stages2")
        reached.add(f"halo.{d}d")
        reached.add(f"halo.pad{pad}")
        if crop is not None:
            reached.add("halo.crop")
    elif fam == "flat":
        reached.add({"f32": "flat.f32", "q1": "flat.q1", "q4": "flat.q4"}.get(case.dtype, "flat.other"))
        if (_knob(case, "flat_ctas") or 1) > 1 and r["grid"] > sms:
            reached.add("flat.ctas")
        if r["stages"] == 2 and _knob(case, "flat_stages") == 2:
            reached.add("flat.stages2")
        if r["warps"] == 1:
            reached.add("flat.warps1")
        if r["table"] == 0 and C > 512:
            reached.add("flat.no_table")
    if op == 2:
        if r["slots"] >= 8 * r["warps"] and _knob(case, "chunk_planes") == 1:
            reached.add("pass2.many_slots")
        if case.fused and r["units"] > 1:
            reached.add("pass2.fused")
    return reached


def _case_regimes(lib, steering, case, sms):
    """Every regime the case reaches over its paddings, crops and forced phases (asserting the family of each)."""
    w = _weights(case, np.random.default_rng(0))
    steering(case.path, case.knobs)
    reached = set()
    for pad in case.pads:
        for crop in case.crops:
            for phase, op in _phases(case):
                r = _route(lib, case, pad, crop, op)
                assert r["path"] == case.path, (case.name, pad, crop, phase, r)
                reached |= _regimes(case, pad, crop, phase, op, r, w, sms)
    return reached


def _gw_close(gw, gw64):
    """grad_weight against the fp64 oracle: rtol 1e-5, atol 1e-5 * max|gw|; a 16-bit grad_weight (same-dtype 16-bit
    layers) is the fp64 sum rounded once to its type, so half an ulp of that type is added to the relative bound."""
    rtol = 1e-5 + (torch.finfo(gw.dtype).eps / 2 if gw.dtype in (torch.float16, torch.bfloat16) else 0.0)
    gw64 = torch.from_numpy(gw64)
    scale = float(gw64.abs().max())
    return torch.allclose(gw.double(), gw64, rtol=rtol, atol=1e-5 * scale + 1e-30)


def _run_float(case, pad, crop, w, rng, dev, lib, oracle, steering):
    from torchshifts import functional as F
    func = {1: F.shift1d_func, 2: F.shift2d_func, 3: F.shift3d_func}[case.dim]
    sdt, wdt = DTYPES[case.dtype][:2]
    active = case.kind == "active"
    _, lb, rb = _geometry(case, crop)
    oshape = list(case.shape[:2]) + [rb[a] - lb[a] for a in range(case.dim)]
    x = torch.from_numpy(rng.standard_normal(case.shape)).to(sdt)
    g = torch.from_numpy(rng.standard_normal(oshape)).to(sdt)
    wt = torch.from_numpy(w).to(wdt)
    # what the kernels see, in the oracle's types: fp64 layers in fp64, everything else in fp32
    odt = np.float64 if case.dtype == "f64" else np.float32
    xr, gr, wr = (np.ascontiguousarray(t.to(torch.float64).numpy().astype(odt)) for t in (x, g, wt))
    xd, wd = x.to(dev).requires_grad_(True), wt.to(dev).requires_grad_(True)
    b = torch.tensor(crop, dtype=torch.long) if crop is not None else None
    steering(case.path if "fwd" in case.ops else 0, case.knobs)
    if case.fused:
        from torchshifts.sharded import FusedGradWeightAllReduce
        ctx = FusedGradWeightAllReduce(capacity=max(512, case.shape[1] * case.dim), device=dev)
    else:
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        y = func(xd, wd, pad, active, b)
        torch.cuda.synchronize()
        if "fwd" in case.ops:
            assert lib.ts_last_kernel_path() == case.path, case.name
        lib.ts_set_kernel_path(case.path if "bwd" in case.ops else 0)
        y.backward(g.to(dev))
        torch.cuda.synchronize()
    lib.ts_set_kernel_path(0)
    what = (case.name, pad, crop)
    y_ref = torch.from_numpy(oracle.forward(xr, wr, pad, active, crop)).to(sdt)
    gi_ref = torch.from_numpy(oracle.backward(gr, xr, wr, pad, active, crop)[0]).to(sdt)
    _, gw64 = oracle.backward(gr.astype(np.float64), xr.astype(np.float64), wr.astype(np.float64), pad, active, crop)
    assert y.dtype == sdt and xd.grad.dtype == sdt and wd.grad.dtype == wdt
    assert torch.equal(y.detach().cpu(), y_ref), ("forward",) + what
    assert torch.equal(xd.grad.cpu(), gi_ref), ("grad_input",) + what
    assert _gw_close(wd.grad.cpu(), gw64), ("grad_weight",) + what
    return y.detach().cpu(), xd.grad.cpu(), wd.grad.cpu()


def _run_quant(case, pad, crop, w, rng, dev, lib, oracle, steering):
    from torchshifts.quantized.modules.shifts import quantize_shift_weights
    qdt = DTYPES[case.dtype][0]
    if qdt == torch.qint32:
        xq = torch.quantize_per_tensor(torch.from_numpy(rng.standard_normal(case.shape).astype(np.float32)), 1e-6, 0, qdt)
    else:
        xq = torch.quantize_per_tensor(torch.from_numpy(rng.random(case.shape).astype(np.float32)), 1 / 255., 0, qdt)
    qw = quantize_shift_weights(torch.from_numpy(w))
    raw, wzp = quantize_shift_weights_np(w)
    b = torch.tensor(crop, dtype=torch.long) if crop is not None else torch.Tensor()
    steering(case.path, case.knobs)
    yq = getattr(torch.ops.torchshifts, f"shift{case.dim}d")(xq.to(dev), qw.to(dev), b, pad, False)
    torch.cuda.synchronize()
    assert lib.ts_last_kernel_path() == case.path, case.name
    lib.ts_set_kernel_path(0)
    ref = oracle.qforward(xq.int_repr().numpy(), raw, wzp, 0, pad, crop)
    assert np.array_equal(yq.int_repr().cpu().numpy(), ref), (case.name, pad, crop)
    return torch.from_numpy(yq.int_repr().cpu().numpy()), None, None


def _run(case, pad, crop, dev, lib, oracle, steering, seed=1):
    rng = np.random.default_rng(seed)
    w = _weights(case, np.random.default_rng(0))
    fn = _run_quant if case.kind == "quant" else _run_float
    return fn(case, pad, crop, w, rng, dev, lib, oracle, steering)


# ------------------------------------------------------------------------------------------ CPU
def test_debug_route_argument_checks(lib):
    """ts_debug_route validates its arguments before it looks for a device: a bad op, dtype or n_out is
    TS_ERR_INVALID_ARGUMENT on any machine; a valid call needs the device (TS_ERR_NO_DEVICE without one)."""
    from torchshifts._cabi import make_geometry
    geo = make_geometry(2, (2, 8, 16, 32), (8 * 512, 512, 32, 1), [0, 0, 0], [16, 32, 1])
    out = (ct.c_int64 * N_OUT)()
    for op, dtype, eb, n in ((3, 0, 4, N_OUT), (-1, 0, 4, N_OUT), (0, 7, 4, N_OUT), (0, 0 | TS_WEIGHTS_F32, 4, N_OUT),
                             (1, -1, 1, N_OUT), (2, -1, 4, N_OUT), (0, 0, 4, N_OUT - 1), (2, 0, 4, 0)):
        assert lib.ts_debug_route(ct.byref(geo), op, dtype, eb, 0, 0, out, n) == TS_ERR_INVALID_ARGUMENT, (op, dtype, eb, n)
    assert lib.ts_debug_route(ct.byref(geo), 0, 0, 4, 0, 0, None, N_OUT) == TS_ERR_INVALID_ARGUMENT
    want = TS_OK if torch.cuda.is_available() else TS_ERR_NO_DEVICE
    for op, dtype, eb in ((0, 0, 4), (1, 0, 4), (2, 0, 4), (0, -1, 1), (2, 3 | TS_WEIGHTS_F32, 2)):
        assert lib.ts_debug_route(ct.byref(geo), op, dtype, eb, 0, 1, out, N_OUT) == want, (op, dtype)


def test_weights_cover_every_residue():
    """The generated weights reach every residue of the last-axis integer shift modulo the item width (sparse and
    active split), in every case that has at least two channels per residue."""
    for case in CASES:
        item = _item(case)
        if case.weights or case.shape[1] < 2 * item + 2:
            continue
        w = _weights(case, np.random.default_rng(0))[:, -1]
        for iw in (np.rint(w), np.floor(w)):
            assert set(iw.astype(np.int64) % item) == set(range(item)), case.name


def test_cases_claim_only_listed_regimes():
    claimed = {c for case in CASES for c in case.claims}
    assert claimed <= set(REQUIRED), sorted(claimed - set(REQUIRED))
    assert not set(REQUIRED) - claimed, sorted(set(REQUIRED) - claimed)
    assert len({case.name for case in CASES}) == len(CASES)


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_regime_vs_oracle(dev, lib, oracle_port, steer, case):
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    reached = _case_regimes(lib, steer, case, sms)
    missing = set(case.claims) - reached
    assert not missing, f"{case.name} no longer reaches {sorted(missing)} (reached {sorted(reached)})"
    for pad in case.pads:
        for crop in case.crops:
            _run(case, pad, crop, dev, lib, oracle_port, steer)


# One geometry per family, each knob that must not change a result.  y and grad_input are computed element by element:
# bit-identical under every knob.  grad_weight: partial slots are indexed by (chunk, warp), never by CTA, and in the TMA
# and halo families a warp walks its unit's items in a fixed order whatever CTA runs the unit and however deep the ring
# is, so it is bit-identical too -- as long as the plan keeps its images per stage, images per unit and warps.  Two
# exceptions the code shows, where only y and grad_input are compared:
# * a ring-depth knob can lower the stage target (the TMA and staged planners fit `stages` stages into shared memory),
#   which changes the images per stage and so the chunks the partials are grouped by;
# * the staged family deals each stage's edge items to its threads from a running offset kept for the CTA's whole
#   lifetime (EdgeRotor, ts_staged.cu), so which warp sums an edge item depends on the units the CTA ran before: the
#   unit order changes the per-warp sums (each within rounding of the others).
# (ctas_per_sm acts on the staged gather only; the flat family is a forward only.)
INVARIANCE = [
    (Case("inv_tma", TMA, "active", "f32", (6, 300, 12, 64)), ("", "unit_order=0", "tma_stages=2", "tma_stages=7,unit_order=0")),
    (Case("inv_staged", STAGED, "active", "f32", (6, 300, 5, 8, 16), pads=(3,)), ("", "unit_order=0", "stages=2", "stages=8")),
    (Case("inv_staged_gather", STAGED, "sparse", "f32", (6, 300, 8, 40), pads=(2,), ops=("fwd",)),
     ("", "unit_order=0", "stages=2", "ctas_per_sm=3", "stages=7,ctas_per_sm=2,unit_order=0")),
    (Case("inv_halo", HALO, "active", "f32", (6, 300, 20, 24), pads=(3,)), ("", "unit_order=0", "halo_stages=2", "halo_stages=6")),
    (Case("inv_flat", FLAT, "sparse", "f32", (6, 100, 8, 24), ops=("fwd",)), ("", "flat_stages=2", "flat_ctas=3", "flat_ctas=2,flat_stages=3")),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case,variants", INVARIANCE, ids=[c.name for c, _ in INVARIANCE])
def test_knobs_leave_results_bit_identical(dev, lib, oracle_port, steer, case, variants):
    results, plans = [], []
    for knobs in variants:
        case.knobs = knobs
        try:
            steer(case.path, knobs)
            routes = [_route(lib, case, case.pads[0], None, op) for _, op in _phases(case)]
            assert all(r["path"] == case.path for r in routes), (case.name, knobs)
            plans.append([(r["np"], r["npu"], r["warps"], r["slots"]) for r in routes])
            results.append(_run(case, case.pads[0], None, dev, lib, oracle_port, steer))
        finally:
            case.knobs = ""
    compared = 0
    for knobs, plan, res in zip(variants[1:], plans[1:], results[1:]):
        for k, (a, b, what) in enumerate(zip(results[0], res, ("y", "grad_input", "grad_weight"))):
            if a is None:
                continue
            if what == "grad_weight":
                if plan != plans[0] or (case.path == STAGED and "unit_order=0" in knobs):
                    continue
                compared += 1
            assert torch.equal(a, b), (case.name, knobs, what)
    if case.kind != "quant" and "bwd" in case.ops:
        assert compared >= 1, f"{case.name}: no variant kept the plan, grad_weight was never compared"


@pytest.mark.gpu
def test_every_listed_regime_is_reached(dev, lib, steer):
    """What the cases reach, read from their plans: every regime of REQUIRED is claimed by a case that reaches it."""
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    reached = set()
    for case in CASES:
        reached |= _case_regimes(lib, steer, case, sms) & set(case.claims)
    missing = sorted(set(REQUIRED) - reached)
    print(f"[plan regimes] {len(reached)} of {len(REQUIRED)} reached")
    assert not missing, missing
