"""The ahead-of-time kernels (build.py MODELS -> csrc/generated/<model>_<algo>.cu) off their happy path.

Every slot of a model's kernel table (runtime/registry.h, AlgoKernels::f64[4] / f32[4]) is one of three launchers of
kernels/batched_kernel.cuh: launchBatchedTma (bulk-copy tiles), launchBatched<..., STAGED> (software-staged tiles or
direct global I/O) and, behind both, launchSlowPass (flagged tiles). Each has a second path besides its fast one. These
tests run every slot on it:

  * CPU: the slot table parsed from the generated sources agrees with build.MODELS (variant count, CTA size and count,
    a direct-I/O fallback only where the tiles do not fit an SM, FP32 slots exactly for the FP32-built models), and
    every slot is in the GPU matrix below.
  * GPU, per (model, entry point, precision) and kernel variant (GRBDA_KERNEL_VARIANT):
      - odd last tiles: B = 1, 2, 3, 5, 33, BLOCK - 1, BLOCK + 1, 2 BLOCK + 3, 3 BLOCK + 5;
      - flagged tiles: whole turns beyond the fast sin/cos range in tiles 0 and 2, a canonical NaN in tile 2, a large
        angle inside the range in tile 1; outputs prefilled with a sentinel, so a tile nobody wrote shows;
      - inputs at an element offset (not 16-byte aligned: the bulk-copy shell drops to the staged kernel);
      - outputs inside sentinel guard bands through the C ABI at the smallest offsets the ABI admits, and a large
        output at an 8-byte offset refused without a launch.
  * GPU: constraintViolation off the constraint manifold against a numpy replay of the phi program.
References: the oracle (FP64; FP32 on float-rounded inputs) and tests/tape.py.
"""
import ctypes as C
import importlib.util
import math
import os
import re
from collections import namedtuple
from fractions import Fraction

import numpy as np
import pytest

from tape import load_tape, run_tape
from test_gpu_jit_edges import SENTINEL, _check_guards, _guarded, _large, _unaligned
from test_gpu_parity import TOL32, TOL64, oracle_for, relrows

HERE = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(os.path.dirname(HERE), "generalized_rbda_b200")


def _build_module():
    spec = importlib.util.spec_from_file_location("grbda_build_table", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


BUILD = _build_module()
N_MAX = 3 * 128 + 5
TURNS = 4.0e11                            # FP64 whole turns: 2.5e12 rad, beyond the range check (1e12)
IN_RANGE = {"f64": 1.0e8, "f32": 1.0e3}   # large, but inside the fast range
EPS32 = float(np.finfo(np.float32).eps)
PATTERN64 = int(np.array([SENTINEL]).view(np.int64)[0])
PATTERN32 = 0x7FC1CAFE                    # a quiet NaN no kernel computes (CUDA's canonical NaN is 0x7FFFFFFF)
# FP32 slots that no entry point launches: the C ABI has no FP32 constraint violation or external-force dynamics
UNREACHABLE = {("phi", "f32"), ("gfa", "f32"), ("gfs", "f32")}

# FP32 forward dynamics whose error is not that of the solve of H: the four-bar has one reduced coordinate (H is 1 x 1,
# cond(H) = 1), and its explicit form G = [1; -Kd^-1 Ki] solves with the Jacobian Kd of the loop's dependent coordinates.
# Neither cond(H) nor cond(H) cond(Kd) bounds its error (measured on a B200 at 1000 W: up to 10 eps32 cond(H) cond(Kd)).
# Its states are held to a median of 1e-5 and a largest error of 10 x TOL32: near a singular loop configuration the
# FP32 articulated-body slot 0 misses the north-star bound of 1e-4 (2.3e-4 on one of 389 states).
FD32_LOOP_BOUND = {"four_bar"}

_PI = Fraction("3.14159265358979323846264338327950288419716939937510582097494459230781640628620899863")


def _fast_residual(x, prec):
    """|r| of the fast sin/cos reduction (kernels/batched_kernel.cuh, grbda_sincos<true>) at x, computed exactly:
    t = x c + K rounded once to the precision (one FMA), k = t - K, r = x - k pi/2. The polynomials that follow are
    meant for |r| <= pi/4; k is exact up to ~3.5e15 rad (FP64) and ~6.6e6 rad (FP32), far beyond the range check."""
    bits, c, K = (52, 0.63661977236758138, 1.5 * 2.0 ** 52) if prec == "f64" else \
        (23, float(np.float32(0.636619772)), 1.5 * 2.0 ** 23)
    v = Fraction(x) * Fraction(c) + Fraction(K)
    S = Fraction(2) ** (math.floor(math.log2(abs(float(v)))) - bits)
    t = round(v / S) * S
    return abs(Fraction(x) - (t - Fraction(K)) * _PI / 2)


def _beyond_fast_range(prec, sign):
    """an angle (1e18 rad in FP64, 1e9 in FP32) at which the fast reduction leaves |r| >= 16: the fast forms give
    meaningless values there, so only the flagged-tile pass (library sin/cos) can match the reference"""
    dt = np.float64 if prec == "f64" else np.float32
    x = dt(sign * (1.0e18 if prec == "f64" else 1.0e9))
    while _fast_residual(float(x), prec) < 16:
        x = np.nextafter(x, dt(sign * np.inf))
    return float(x)


BEYOND = {prec: (_beyond_fast_range(prec, 1), _beyond_fast_range(prec, -1)) for prec in ("f64", "f32")}

Slot = namedtuple("Slot", "kind block min_blocks body")


# ---- the slot table of the build ----------------------------------------------------------------------------
def _ident(name):
    return "".join(c if c.isalnum() else "_" for c in name)


def _shape_constants():
    text = open(os.path.join(PKG, "csrc", "kernels", "shapes.h")).read()
    return {k: int(a) * int(b) for k, a, b in re.findall(r"constexpr size_t (\w+) = (\d+) \* (\d+);", text)}


_SLOT = re.compile(r"&launchBatched(Tma)?<(double|float), (Body\d+), (\d+), (\d+)(?:, (true|false))?>|nullptr")
_TABLE = re.compile(r"k_algo = \{\s*\{(.*?)\},\s*\{(.*?)\},\s*\{(\d+), (\d+), (\d+)\}, \{(\d+), (\d+), (\d+)\}", re.S)
_BODY = re.compile(r"struct (Body\d+)\s*\{.*?RANGE_CHECKED = (true|false);.*?STAGE_BUFFERS = (\d+);.*?PARKED = (true|false);"
                   r".*?PARK_EXTRA = (\d+);.*?DIRECT_OUT0 = (true|false);", re.S)


def _parse_slots(text):
    slots = []
    for tma, _, body, block, ctas, staged in _SLOT.findall(text):
        if not body:
            slots.append(None)
        else:
            slots.append(Slot("T" if tma else ("S" if staged == "true" else "D"), int(block), int(ctas), body))
    assert len(slots) == 4, text
    return slots


_TABLE_CACHE = {}


def slot_table(gen_dir=None):
    """{(model, algo): dict(f64=[Slot | None] * 4, f32=[...], n_in, n_out, bodies={name: constants})}, or None for an
    entry point whose file modelc did not write (a phi program without implicit clusters)."""
    gen_dir = gen_dir or BUILD.GEN
    if gen_dir in _TABLE_CACHE:
        return _TABLE_CACHE[gen_dir]
    table = {}
    for model, (algos, _, _) in BUILD.MODELS.items():
        for algo in algos.split(","):
            if algo == "gen":
                continue
            path = os.path.join(gen_dir, "%s_%s.cu" % (_ident(model), algo))
            if not os.path.exists(path):
                table[(model, algo)] = None
                continue
            text = open(path).read()
            t = _TABLE.search(text)
            assert t, path
            bodies = {b: dict(range_checked=r == "true", stage_buffers=int(s), parked=p == "true", park_extra=int(e),
                              direct=d == "true") for b, r, s, p, e, d in _BODY.findall(text)}
            table[(model, algo)] = dict(f64=_parse_slots(t.group(1)), f32=_parse_slots(t.group(2)),
                                        n_in=[int(x) for x in t.group(3, 4, 5)],
                                        n_out=[int(x) for x in t.group(6, 7, 8)], bodies=bodies)
    _TABLE_CACHE[gen_dir] = table
    return table


def _variant_specs(model, algo):
    """build.MODELS' variants of one entry point: [(kind, block, min_blocks, keywords)]"""
    segs = dict(seg.split("=", 1) for seg in BUILD.MODELS[model][1].split("|"))
    out = []
    for v in segs[algo].split(";"):
        p = v.split(",")
        out.append((p[0], int(p[1]), int(p[2]), {k for k in p[3:] if not k.isdigit()}))
    return out


def _tile_bytes(kind, n_in, n_out, stage_buffers, block, elem, park_extra, direct):
    """kernels/shapes.h shapeTileBytes (kind S) / shapeTmaBytes (kind T), with the park area and direct output 0."""
    a16 = lambda x: (x + 15) & ~15  # noqa: E731
    chunked = n_out[0] > 64 or n_out[1] > 16 or n_out[2] > 16
    stage = (stage_buffers * block * 17 * elem if chunked else 0) + (block * (park_extra | 1) * elem if park_extra else 0)
    small_out0 = n_out[0] <= 64 and not direct
    if kind == "S":
        elems = sum((n | 1) * block for n in n_in if n) + ((n_out[0] | 1) * block if small_out0 else 0)
        return a16(elems * elem) + stage
    stride = lambda n: n + 16 // elem if n >= 12 and (n * elem) % 16 == 0 else n  # noqa: E731
    off = 16
    for n in n_in:
        off = a16(off + stride(n) * block * elem)
    off = a16(off + (stride(n_out[0]) * block * elem if small_out0 else 0))
    return off + stage


# ---- the GPU matrix: (model, algo, precision) -> the entry point that launches the slot --------------------------
Entry = namedtuple("Entry", "algos inputs shapes call cabi")
ENTRIES = {
    "id": Entry(("id",), ("q", "yd", "aux"), lambda m: [(m.nv,)],
                lambda m, a, o: [m.inverseDynamics(a["q"], a["yd"], a["aux"], out=o[0])], "grbda_cuda_inverse_dynamics_%s"),
    "fd": Entry(("fd",), ("q", "yd", "aux"), lambda m: [(m.nv,)],
                lambda m, a, o: [m.forwardDynamics(a["q"], a["yd"], a["aux"], out=o[0])], "grbda_cuda_forward_dynamics_%s"),
    "fk": Entry(("fk",), ("q", "yd"), lambda m: [(m.nb, 3), (m.nb, 3, 3), (m.nb, 6)],
                lambda m, a, o: list(m.forwardKinematics(a["q"], a["yd"], out=tuple(o))),
                "grbda_cuda_forward_kinematics_%s"),
    "h": Entry(("h",), ("q",), lambda m: [(m.nv, m.nv)], lambda m, a, o: [m.getMassMatrix(a["q"], out=o[0])],
               "grbda_cuda_mass_matrix_%s"),
    # external forces: ID then tau - J^T f (gfs); tau + J^T f (gfa) then FD. GRBDA_KERNEL_VARIANT selects both slots.
    "gfs": Entry(("id", "gfs"), ("q", "yd", "aux", "f"), lambda m: [(m.nv,)],
                 lambda m, a, o: [m.inverseDynamics(a["q"], a["yd"], a["aux"], out=o[0], f_ext=a["f"])],
                 "grbda_cuda_inverse_dynamics_ext_%s"),
    "gfa": Entry(("gfa", "fd"), ("q", "yd", "aux", "f"), lambda m: [(m.nv,)],
                 lambda m, a, o: [m.forwardDynamics(a["q"], a["yd"], a["aux"], out=o[0], f_ext=a["f"])],
                 "grbda_cuda_forward_dynamics_ext_%s"),
}
GPU_CASES = [(model, algo, prec) for model, (algos, _, f32) in BUILD.MODELS.items() for algo in algos.split(",")
             if algo in ENTRIES for prec in ("f64", "f32")
             if prec == "f64" or (f32 and (algo, prec) not in UNREACHABLE)]
PHI_MODELS = [model for model, (algos, _, _) in BUILD.MODELS.items() if "phi" in algos.split(",")]


def _variants(table, model, algo, prec):
    """variant indices at which every slot the entry point launches exists"""
    rows = [table[(model, a)][prec] for a in ENTRIES[algo].algos]
    return [v for v in range(4) if all(r[v] is not None for r in rows)]


# ---- CPU ------------------------------------------------------------------------------------------------------
def test_slot_table_agrees_with_the_build(grbda, tmp_path):
    table = slot_table()
    consts = _shape_constants()
    sm, slow_limit = consts["SM_SHARED_BYTES"], consts["SLOW_PASS_STAGED_LIMIT"]
    fallbacks = []
    for model, (algos, _, f32) in BUILD.MODELS.items():
        for algo in (a for a in algos.split(",") if a != "gen"):
            t = table[(model, algo)]
            if t is None:
                # modelc writes no phi program for a model without implicit clusters: its phi program is empty
                assert algo == "phi", (model, algo)
                h = grbda.ClusterTreeModel.from_robot(model, device=None)
                h.dump_program(grbda.ALGO_PHI, str(tmp_path / "phi.tape"))
                assert len(load_tape(str(tmp_path / "phi.tape"))["outs"][0]) == 0, model
                continue
            specs = _variant_specs(model, algo)
            n_in, n_out = t["n_in"], t["n_out"]
            park_extra = max(b["park_extra"] for b in t["bodies"].values())
            stage_buffers = t["bodies"][t["f64"][0].body]["stage_buffers"]
            chunked = n_out[0] > 64 or n_out[1] > 16 or n_out[2] > 16
            for prec, elem in (("f64", 8), ("f32", 4)):
                slots = t[prec]
                what = "%s/%s/%s" % (model, algo, prec)
                if prec == "f32" and not f32:
                    assert slots == [None] * 4, what
                    continue
                assert slots == [s for s in slots if s] + [None] * (4 - len(specs)), what
                for v, ((kind, block, ctas, kw), s) in enumerate(zip(specs, slots)):
                    assert (s.block, s.min_blocks) == (block, ctas), (what, v, s)
                    body = t["bodies"][s.body]
                    # (an FP32 launcher of a parked variant gets the unparked body, which keeps its output tile)
                    assert body["direct"] == ("direct" in kw) or (prec == "f32" and not body["direct"]), (what, v)
                    assert not body["parked"] or (prec == "f64" and "park" in kw), (what, v)
                    # modelc: parking only where the flagged-tile pass stages the rows too, and for large outputs
                    # only from 400 values on; FP32 bodies are never parked
                    park = prec == "f64" and "park" in kw and \
                        _tile_bytes("S", n_in, n_out, 3, block, 8, 0, "direct" in kw) <= slow_limit and \
                        not ((algo == "h" or chunked) and max(n_out) < 400)
                    fits = kind == "D" or _tile_bytes(kind, n_in, n_out, stage_buffers, block, elem,
                                                      park_extra if park else 0, "direct" in kw) + 1024 <= sm
                    assert s.kind == (kind if fits else "D"), (what, v, kind, s)
                    if s.kind != kind:
                        fallbacks.append("%s variant %d" % (what, v))
    print("direct-I/O fallbacks:", ", ".join(fallbacks) or "none")


def test_every_slot_is_in_the_gpu_matrix(grbda):
    """A slot that build.py adds is tested by the GPU matrix without editing this file; an FP32 slot without an entry
    point is the only one left out."""
    table = slot_table()
    cases = set(GPU_CASES)
    covered = set()
    for model, algo, prec in GPU_CASES:
        vs = _variants(table, model, algo, prec)
        assert vs and vs[0] == 0, (model, algo, prec)
        covered |= {(model, a, prec, v) for a in ENTRIES[algo].algos for v in vs}
    for (model, algo), t in table.items():
        if t is None:
            continue
        for prec in ("f64", "f32"):
            for v, s in enumerate(t[prec]):
                if s is None or (algo, prec) in UNREACHABLE:
                    continue
                if algo == "phi":  # test_constraint_violation_off_the_manifold runs every phi variant
                    assert model in PHI_MODELS
                    continue
                assert (model, algo, prec) in cases and (model, algo, prec, v) in covered, (model, algo, prec, v)


# ---- GPU helpers ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _filled(torch, shape, prec):
    """an output prefilled with the sentinel"""
    if prec == "f64":
        return torch.full(shape, SENTINEL, dtype=torch.float64, device="cuda")
    return torch.full(shape, PATTERN32, dtype=torch.int32, device="cuda").view(torch.float32)


def _sentinels(torch, t):
    bits = t.view(torch.int64 if t.dtype == torch.float64 else torch.int32)
    return int((bits == (PATTERN64 if t.dtype == torch.float64 else PATTERN32)).sum())


def _unaligned_f32(torch, t):
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    u = buf[1:].view(t.shape)
    u.copy_(t)
    assert u.data_ptr() % 16 == 4
    return u


def _guarded_f32(torch, shape, large, front=None):
    """FP32 counterpart of _guarded: a large output at a 16-byte offset, a small one at 4 bytes"""
    n = int(np.prod(shape))
    front = (4 if large else 1) if front is None else front
    buf = torch.full((front + n + 64,), PATTERN32, dtype=torch.int32, device="cuda").view(torch.float32)
    return buf, buf[front:front + n].view(shape), front, n


def _check_guards_f32(torch, guarded):
    for buf, _, front, n in guarded:
        bits = buf.view(torch.int32).cpu().numpy()
        assert (bits[:front] == PATTERN32).all() and (bits[front + n:] == PATTERN32).all(), "write outside the output"
        assert not (bits[front:front + n] == PATTERN32).any(), "output element not written"


def _coordinates(m, prec):
    """(c0, c1, plain): the coordinates that get angles beyond the range check in tiles 0 and 2. plain: joints of
    explicit clusters without a rotor body, which get angles beyond the range where the fast reduction is exact
    (BEYOND). A geared rotor multiplies such an angle, and the kernel and the oracle may round that product
    differently, so models without such a joint get FP64 whole turns (2.5e12 rad) on a one-coordinate cluster, or on a
    loop cluster, and no FP32 angles. Those cases show that the flagged tiles are recomputed and written; the fast
    forms are still exact at 2.5e12 rad, so the launch count shows that the flagged-tile pass ran."""
    cl = [c for c in m.clusters() if c["type"] != 0]
    plain = [c["position_index"] for c in cl if c["type"] == 2 and c["num_bodies"] == c["num_positions"]]
    if plain:
        return plain[0], plain[-1], True
    if prec == "f32":
        return None
    ones = [c["position_index"] for c in cl if c["type"] == 2 and c["num_positions"] == 1]
    ones = ones or [c["position_index"] for c in cl]
    return ones[0], ones[-1], False


_CTX = {}


def _context(grbda, oracle, torch, name):
    """The model, its N_MAX generated states and external forces, and references computed once (sliced per case)."""
    if name in _CTX:
        return _CTX[name]
    m = grbda.ClusterTreeModel.from_robot(name)
    o = oracle_for(oracle, m, name)
    q, yd, aux, flags = m.generateStates(N_MAX, seed=37)
    assert int(flags.sum()) == 0
    bodies = m.externalForceBodies()
    gen = torch.Generator(device="cuda").manual_seed(41)
    f = (torch.rand((N_MAX, len(bodies), 6), dtype=torch.float64, device="cuda", generator=gen) - 0.5) * 40.0
    ins = {"f64": dict(q=q, yd=yd, aux=aux, f=f), "f32": dict(q=q.float(), yd=yd.float(), aux=aux.float())}
    ctx = dict(name=name, m=m, o=o, bodies=bodies, inputs=ins, refs={}, nan_coordinate={})
    _CTX[name] = ctx
    return ctx


def _reference(ctx, algo, a):
    """oracle outputs [B, n] of an entry point on the (float-rounded) inputs a (torch tensors); for FD also the
    condition number of H per state"""
    o = ctx["o"]
    q, yd, aux = (a[k].double().cpu().numpy() for k in ("q", "yd", "aux"))
    B = len(q)
    if algo == "id":
        outs = [o.inverse_dynamics(q, yd, aux)]
    elif algo == "fd":
        outs = [o.forward_dynamics(q, yd, aux)]
    elif algo == "h":
        outs = [o.mass_matrix(q)]
    elif algo == "fk":
        outs = list(o.forward_kinematics(q, yd))
    else:
        f_full = np.zeros((B, o.nb, 6))
        f_full[:, ctx["bodies"], :] = a["f"].cpu().numpy()
        outs = [o.dynamics_with_external_forces(q, yd, aux, f_full, forward=algo == "gfa")]
    cond = np.linalg.cond(o.mass_matrix(q)) if algo == "fd" else None
    return [np.asarray(r).reshape(B, -1) for r in outs], cond


def _full_reference(ctx, algo, prec):
    if (algo, prec) not in ctx["refs"]:
        ctx["refs"][(algo, prec)] = _reference(ctx, algo, ctx["inputs"][prec])
    return ctx["refs"][(algo, prec)]


def _check(algo, prec, v, outs, want, cond, rows, what):
    """FP64: 1e-10 per state. FP32 on float-rounded inputs: ID / H / FK 1e-4 per state; FD the bound of a backward
    stable solve, err <= 2 eps32 cond(H) per state (the factorising slots lose up to ~1e-4 on the 16-link chain), and
    on slot 0, the articulated-body sweep that ships, also 1e-4. FD32_LOOP_BOUND: see there."""
    got = [t.double().cpu().numpy().reshape(t.shape[0], -1)[rows] for t in outs]
    want = [w[rows] for w in want]
    if prec == "f32" and algo == "fd":
        g, w = got[0], want[0]
        err = np.abs(g - w).max(1) / np.abs(w).max(1)
        if (what[0] if isinstance(what, tuple) else what).split("/")[0] in FD32_LOOP_BOUND:
            assert err.max() < 10 * TOL32 and np.median(err) < 1e-5, (what, err.max(), np.median(err))
            return
        assert (err / (2.0 * EPS32 * cond[rows])).max() < 1.0, (what, "err / (2 eps32 cond(H))")
        if v == 0:
            assert err.max() < TOL32, (what, "north-star bound", err.max())
        return
    tol = TOL64 if prec == "f64" else TOL32
    for k, (g, w) in enumerate(zip(got, want)):
        assert relrows(g, w) < tol, (what, "output %d" % k, relrows(g, w))


def _nan_coordinate(ctx, algo, prec):
    """the last coordinate the entry point's outputs depend on (the first joint of a fixed base does not enter H, nor,
    in a planar model, the dynamics): a NaN there must reach the state's outputs"""
    if (algo, prec) in ctx["nan_coordinate"]:
        return ctx["nan_coordinate"][(algo, prec)]
    a = {k: t[:1] for k, t in ctx["inputs"][prec].items()}
    base = _reference(ctx, algo, a)[0]
    for c in reversed(range(a["q"].shape[1])):
        ap = dict(a)
        ap["q"] = a["q"].clone()
        ap["q"][0, c] += 0.5
        if any(np.abs(x - y).max() > 1e-6 * max(1.0, np.abs(y).max()) for x, y in zip(_reference(ctx, algo, ap)[0], base)):
            ctx["nan_coordinate"][(algo, prec)] = c
            return c
    raise AssertionError("no coordinate changes the outputs")


def _slice(a, n):
    return {k: t[:n] for k, t in a.items()}


def _guards_ok(torch, guarded, prec, what):
    try:
        (_check_guards if prec == "f64" else _check_guards_f32)(torch, guarded)
    except AssertionError as e:
        raise AssertionError("%s: %s" % (what, e)) from e


# ---- GPU: every slot off its happy path -----------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,algo,prec", GPU_CASES, ids=["%s-%s-%s" % c for c in GPU_CASES])
def test_every_slot_off_its_happy_path(grbda, oracle, torch, name, algo, prec, monkeypatch, capsys):
    """Every variant of the slots the entry point launches; the flagged-tile cases of all variants are collected and
    reported together after the others, so that a build without the flagged-tile pass fails there only."""
    table = slot_table()
    ep = ENTRIES[algo]
    ctx = _context(grbda, oracle, torch, name)
    m, inp = ctx["m"], ctx["inputs"][prec]
    ref, cond = _full_reference(ctx, algo, prec)
    shapes = ep.shapes(m)
    rows_of = lambda B: np.arange(B)  # noqa: E731
    L = grbda.lib()
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ran, flagged_failures = [], []

    def call(a, B):
        outs = ep.call(m, a, [_filled(torch, (B,) + s, prec) for s in shapes])
        torch.cuda.synchronize()
        return outs

    for v in _variants(table, name, algo, prec):
        monkeypatch.setenv("GRBDA_KERNEL_VARIANT", str(v))
        slots = [table[(name, a)][prec][v] for a in ep.algos]
        bodies = [table[(name, a)]["bodies"][s.body] for a, s in zip(ep.algos, slots)]
        blocks = sorted({s.block for s in slots})
        label = "%s/%s/%s variant %d [%s]" % (name, algo, prec, v, "; ".join(
            "%s %s,%d,%d" % (a, s.kind, s.block, s.min_blocks) for a, s in zip(ep.algos, slots)))

        # odd last tiles
        sizes = {1, 2, 3, 5, 33}
        for b in blocks:
            sizes |= {b - 1, b + 1, 2 * b + 3, 3 * b + 5}
        for B in sorted(s for s in sizes if s <= N_MAX):
            outs = call(_slice(inp, B), B)
            assert sum(_sentinels(torch, t) for t in outs) == 0, (label, "B=%d" % B, "output not written")
            _check(algo, prec, v, outs, ref, cond, rows_of(B), (label, "B=%d" % B))

        # unaligned inputs: each in turn at one element past a 16-byte boundary
        bk = blocks[-1]
        N = 3 * bk + 5
        a = _slice(inp, N)
        before = grbda.launch_count()
        aligned = call(a, N)
        launches = grbda.launch_count() - before
        for key in ep.inputs:
            au = dict(a)
            au[key] = (_unaligned if prec == "f64" else _unaligned_f32)(torch, a[key])
            before = grbda.launch_count()
            outs = call(au, N)
            assert grbda.launch_count() - before <= launches, (label, "unaligned " + key, "extra launches")
            for k, (g, g0) in enumerate(zip(outs, aligned)):
                d = relrows(g.double().cpu().numpy().reshape(N, -1), g0.double().cpu().numpy().reshape(N, -1))
                assert d < (1e-12 if prec == "f64" else 1e-5), (label, "unaligned " + key, k, d)
            _check(algo, prec, v, outs, ref, cond, rows_of(N), (label, "unaligned " + key))

        # guard bands through the C ABI; the kernel's output k of the last program decides large or small
        fn = getattr(L, ep.cabi % prec)
        widths = [int(np.prod(s)) for s in shapes]
        for B in (1, 2 * bk + 3):
            what = "%s, guard bands B=%d" % (label, B)
            ins = [inp[k][:B] for k in ep.inputs]
            if prec == "f64":
                guarded = [_guarded(torch, (B, n), _large(k, n)) for k, n in enumerate(widths)]
            else:
                guarded = [_guarded_f32(torch, (B, n), _large(k, n)) for k, n in enumerate(widths)]
            status = fn(m._h, *[P(t) for t in ins], *[P(g[1]) for g in guarded], B, st)
            assert status == 0, (what, status, L.grbda_cuda_last_error_string().decode())
            torch.cuda.synchronize()
            _guards_ok(torch, guarded, prec, what)
            _check(algo, prec, v, [g[1] for g in guarded], ref, cond, rows_of(B), what)
        large = [k for k, n in enumerate(widths) if _large(k, n)]
        if large:
            B = 2 * bk + 3
            what = "%s, output %d at an 8-byte offset, B=%d" % (label, large[0], B)
            ins = [inp[k][:B] for k in ep.inputs]
            guarded = []
            for k, n in enumerate(widths):
                if prec == "f64":  # (the small-output placement of _guarded is the 8-byte offset)
                    guarded.append(_guarded(torch, (B, n), _large(k, n) and k != large[0]))
                else:
                    guarded.append(_guarded_f32(torch, (B, n), _large(k, n), 2 if k == large[0] else None))
            assert guarded[large[0]][1].data_ptr() % 16 == 8
            before = grbda.launch_count()
            status = fn(m._h, *[P(t) for t in ins], *[P(g[1]) for g in guarded], B, st)
            assert status == 1, (what, "accepted", status)  # GRBDA_ERR_INVALID_ARGUMENT
            torch.cuda.synchronize()
            assert grbda.launch_count() == before, (what, "launch after a refused call")
            assert sum(_sentinels(torch, g[0]) for g in guarded) == sum(g[0].numel() for g in guarded), \
                (what, "refused call wrote into an output")

        # flagged tiles: 0 and 2 (angles beyond the range check, then a NaN), not 1 (a large angle inside the range)
        try:
            _flagged_tiles(grbda, torch, ctx, algo, prec, v, label, call, a, N, slots, bodies, ref, cond)
        except AssertionError as e:
            flagged_failures.append(str(e))
        ran.append(label)
    with capsys.disabled():
        print("\n" + "\n".join(ran))
    assert not flagged_failures, "\n".join(flagged_failures)


def _flagged_tiles(grbda, torch, ctx, algo, prec, v, label, call, a, N, slots, bodies, ref, cond):
    """Outputs prefilled with the sentinel: the fast kernel leaves a flagged tile unwritten, so a tile without
    sentinels was written by the flagged-tile pass; each call launches the fast kernel and that pass per program."""
    m = ctx["m"]
    bk = max(s.block for s in slots)
    r0, r1, r2, rn = 5, bk + 7, 2 * bk + 5, 2 * bk + 9
    launches = sum(1 + b["range_checked"] for b in bodies)
    base = [t.cpu() for t in call(a, N)]

    def tiles_of(*rs):
        mask = np.zeros(N, dtype=bool)
        for blk in {s.block for s in slots}:
            for r in rs:
                mask[(r // blk) * blk:min(N, (r // blk + 1) * blk)] = True
        return mask

    def same_bits(outs, mask, what):
        sel = torch.from_numpy(mask)
        for k, (g, g0) in enumerate(zip(outs, base)):
            assert torch.equal(g.cpu()[sel], g0[sel]), (label, what, "output %d: unflagged tiles changed" % k)

    def flagged_call(af, what):
        before = grbda.launch_count()
        outs = call(af, N)
        assert sum(_sentinels(torch, t) for t in outs) == 0, (label, what, "flagged tile not written")
        return outs, grbda.launch_count() - before

    def launched(n, what):  # (checked after the values: a wrong value is the more telling failure)
        assert n == launches, (label, what, "launches: %d, fast kernel + flagged-tile pass: %d" % (n, launches))

    coords = _coordinates(m, prec)
    if coords:
        c0, c1, plain = coords
        af = dict(a)
        af["q"] = a["q"].clone()
        what = "angles beyond the fast reduction" if plain else "whole turns"
        if plain:
            af["q"][r0, c0], af["q"][r2, c1] = BEYOND[prec]
        else:
            af["q"][r0, c0] += 2.0 * np.pi * TURNS
            af["q"][r2, c1] -= 2.0 * np.pi * TURNS
        af["q"][r1, c0] += 2.0 * np.pi * IN_RANGE[prec]
        outs, n = flagged_call(af, what)
        pert = [r0, r1, r2]
        ref_p, cond_p = _reference(ctx, algo, {k: t[pert] for k, t in af.items()})
        want = [r[:N].copy() for r in ref]
        cond_w = cond[:N].copy() if cond is not None else None
        for w, rp in zip(want, ref_p):
            w[pert] = rp
        if cond_w is not None:
            cond_w[pert] = cond_p
        flagged = tiles_of(r0, r2)
        _check(algo, prec, v, outs, want, cond_w, np.flatnonzero(flagged), (label, what + ", flagged tiles"))
        _check(algo, prec, v, outs, want, cond_w, [r1], (label, "large angle inside the fast range"))
        keep = ~flagged
        keep[r1] = False
        same_bits(outs, keep, what)
        launched(n, what)
    # a canonical NaN: its state is NaN, the rest of its tile is recomputed from the same inputs
    an = dict(a)
    an["q"] = a["q"].clone()
    an["q"][rn, _nan_coordinate(ctx, algo, prec)] = float("nan")
    outs, n = flagged_call(an, "NaN")
    host = [t.double().cpu().numpy().reshape(N, -1) for t in outs]
    assert any(np.isnan(h[rn]).any() for h in host), (label, "NaN state has no NaN output")
    nan_tile = tiles_of(rn)
    others = np.flatnonzero(nan_tile & (np.arange(N) != rn))
    assert all(np.isfinite(h[others]).all() for h in host), (label, "NaN leaked into other states of its tile")
    _check(algo, prec, v, outs, ref, cond, others, (label, "NaN tile"))
    same_bits(outs, ~nan_tile, "NaN")
    launched(n, "NaN")


# ---- GPU: constraint violation off the manifold -------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", PHI_MODELS)
def test_constraint_violation_off_the_manifold(grbda, torch, name, tmp_path, monkeypatch):
    """max |phi| per state at q + 1e-3 noise against the numpy replay of the phi program, for every phi variant: tail
    sizes, q at an 8-byte offset, the output inside a guard band. A model without implicit clusters has an empty phi
    program: zero."""
    table = slot_table()
    m = grbda.ClusterTreeModel.from_robot(name)
    q, _, _, _ = m.generateStates(N_MAX, seed=43)
    gen = torch.Generator(device="cuda").manual_seed(47)
    q = q + 1e-3 * (torch.rand(q.shape, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1)
    m.dump_program(grbda.ALGO_PHI, str(tmp_path / "phi.tape"))
    phi = run_tape(load_tape(str(tmp_path / "phi.tape")), [q.cpu().numpy()])[0]
    want = np.abs(phi).max(1) if phi.shape[1] else np.zeros(N_MAX)
    t = table[(name, "phi")]
    if t is None:
        assert phi.shape[1] == 0
        variants = [(0, 128)]
    else:
        assert want.min() > 1e-8, "the perturbed states are on the manifold"
        variants = [(v, s.block) for v, s in enumerate(t["f64"]) if s]
    L = grbda.lib()
    for v, block in variants:
        monkeypatch.setenv("GRBDA_KERNEL_VARIANT", str(v))
        label = "%s/phi variant %d" % (name, v)

        def check(got, B, what):
            got = got.cpu().numpy()
            assert got.shape == (B,)
            if t is None:
                assert (got == 0).all(), (label, what)
            else:
                err = np.abs(got - want[:B]) / np.maximum(want[:B], 1e-12)
                assert err.max() < 1e-10, (label, what, err.max())

        for B in sorted(s for s in {1, 2, 3, 5, 33, block - 1, block + 1, 2 * block + 3, 3 * block + 5} if s <= N_MAX):
            check(m.constraintViolation(q[:B]), B, "B=%d" % B)
        check(m.constraintViolation(_unaligned(torch, q)), N_MAX, "q at an 8-byte offset")
        for B in (1, 2 * block + 3):
            what = "%s, guard bands B=%d" % (label, B)
            guarded = [_guarded(torch, (B,), False)]
            status = L.grbda_cuda_constraint_violation_f64(m._h, C.c_void_p(q.data_ptr()),
                                                           C.c_void_p(guarded[0][1].data_ptr()), B,
                                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert status == 0, (what, status)
            torch.cuda.synchronize()
            _guards_ok(torch, guarded, "f64", what)
            check(guarded[0][1], B, what)
