"""The run-time compiled kernels (runtime/jit.cpp, jitLaunch) off their happy path.

Every operational-space, derivative and VJP program, and every program of a model outside build.py's table, is
launched by jitLaunch, which has its own shape choice (chooseShape), alignment rule and flagged-tile pass. These tests
run those programs where they can go wrong quietly:

  * CPU: every launch shell (GRBDA_JIT_SHAPE = D, T,64,2, T,128,1 and the default) compiles to an sm_100a cubin
    for programs 8-18 and FP32 ID / FK / H of a floating-base model.
  * GPU, per model and shell, for every run-time compiled entry point:
      - odd last tiles: B = 1, 2 block + 1, 2 block + 3 and 3 block + 5, against the oracle or the numpy tape replay;
      - flagged tiles: whole turns beyond the fast sin/cos range on two states in tiles 0 and 2; the flagged tiles
        against the reference, every other tile bit for bit equal to the unperturbed call;
      - inputs at an 8-byte offset (the bulk-copy engine needs 16): one slow launch per program of the TMA shell,
        1e-12 against the aligned call and the reference at the existing tolerance.
  * GPU: outputs inside NaN-sentinel guard bands through the C ABI: nothing written outside, everything inside.
  * GPU: FP32 forward kinematics (128-bit ring stores) against the oracle, and FP32 ID / H, at B = 2 * 128 + 3.
"""
import ctypes as C
import os
import re
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from mirror import mirror_to_oracle
from tape import load_tape, run_tape
from test_compiler_cpu import contact_set
from test_gpu_parity import TOL32, TOL64, oracle_for, relrows
from test_vjp import rel

HERE = os.path.dirname(os.path.abspath(__file__))
URDF = os.path.join(HERE, "urdf_corpus", "revolute_rotor_branch_2_3.urdf")  # floating base, nq = 13: not ahead of time
TOL_FD, TOL_OSIM = 1e-9, 1e-8
# forced shells (runtime/jit.cpp chooseShape): direct global I/O, TMA with 64-thread CTAs, TMA with one CTA per SM
SHAPES = ["D", "T,64,2", "T,128,1"]
SM_CTA_SHARED = 227 * 1024  # largest dynamic shared memory one CTA may opt into
TURNS = 4.0e11              # whole turns: 2.5e12 rad, beyond the 1e12 of the fast FP64 reduction


def shape_tma_bytes(n_in, n_out, stage_buffers, block, elem):
    """kernels/shapes.h shapeTmaBytes (no park area)."""
    a16 = lambda x: (x + 15) & ~15  # noqa: E731
    stride = lambda n: n + 16 // elem if n >= 12 and (n * elem) % 16 == 0 else n  # noqa: E731
    off = 16
    for n in n_in:
        off = a16(off + stride(n) * block * elem)
    off = a16(off + (stride(n_out[0]) * block * elem if n_out[0] <= 64 else 0))
    chunked = n_out[0] > 64 or n_out[1] > 16 or n_out[2] > 16
    return off + (stage_buffers * block * 17 * elem if chunked else 0)


def host_model(grbda):
    m = grbda.ClusterTreeModel.from_urdf(URDF, device=None)
    m.setContactPoints(*contact_set(m))
    m.setExternalForceBodies(list(range(m.nb)))
    return m


@pytest.mark.parametrize("shape", SHAPES + [None])
def test_every_shell_compiles_for_sm100a(grbda, shape, tmp_path, monkeypatch):
    """Each shell forced on programs 8-18 (FP64) and ID / FK / H (FP32): an sm_100a cubin, the shell asked for in the
    kernel names, and no vector-store body in a CTA of fewer than 128 threads (one warp per alignment class). A shell
    whose TMA tiles exceed what one CTA may hold is skipped: it could never be launched, so its cubin says nothing."""
    if shape:
        monkeypatch.setenv("GRBDA_JIT_SHAPE", shape)
    else:
        monkeypatch.delenv("GRBDA_JIT_SHAPE", raising=False)
    jobs = [(a, False) for a in range(8, 19)] + [(a, True) for a in (grbda.ALGO_ID, grbda.ALGO_FK, grbda.ALGO_H)]

    def compile_one(job):
        algo, f32 = job
        m = host_model(grbda)  # one handle per thread
        src, cubin = str(tmp_path / ("%d_%d.cu" % job)), str(tmp_path / ("%d_%d.cubin" % job))
        m.jit_compile(algo, f32, src, None)
        text = open(src).read()
        sizes = {k: int(v) for k, v in re.findall(r"\b(N_IN\d|N_OUT\d|STAGE_BUFFERS) = (\d+)", text)}
        block = int(shape.split(",")[1]) if shape and shape[0] == "T" else 128
        tma = shape is None and m.kernel_info(algo, f32)["tma"] or (shape or "").startswith("T")
        n_in = [sizes["N_IN%d" % i] for i in range(3)]
        n_out = [sizes["N_OUT%d" % i] for i in range(3)]
        if tma and shape_tma_bytes(n_in, n_out, sizes["STAGE_BUFFERS"], block, 4 if f32 else 8) > SM_CTA_SHARED:
            return job, text, None
        m.jit_compile(algo, f32, None, cubin)
        return job, text, open(cubin, "rb").read()

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_one, jobs))
    compiled = 0
    for (algo, f32), text, blob in results:
        kernels = re.findall(r"// kernel: (.*)", text)
        if shape == "D":
            assert "grbda_batched_kernel<" in kernels[0] and ", 128, 2, false, true>" in kernels[0]
        elif shape:
            block, ctas = shape.split(",")[1:]
            assert kernels[0].startswith("grbda_kernels::grbda_batched_kernel_tma<") and \
                kernels[0].endswith(", %s, %s>" % (block, ctas)), kernels[0]
            assert len(kernels) == 2  # the flagged-tile / unaligned pass of a TMA shell always exists
            if block != "128":
                assert "VECTOR_STORES = true" not in text
        if blob is None:
            continue
        compiled += 1
        assert blob[:4] == b"\x7fELF" and len(blob) > 10000, (algo, f32)
    assert compiled >= len(jobs) - 2


# ---- GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


class EntryPoint:
    """One run-time compiled entry point: the programs it launches, how to call it on a dict of input tensors, the
    input besides q that the unaligned case offsets, the number of launches besides its programs, its reference."""

    def __init__(self, name, programs, call, ref, tol, second=None, extra=0):
        self.name, self.programs, self.call, self.ref, self.tol = name, programs, call, ref, tol
        self.second, self.extra = second, extra


def _replay(ctx, algo, ins):
    return run_tape(ctx["tape"](algo), ins)


def _id_ext_vjp_ref(ctx, a, g):
    idv = _replay(ctx, g.ALGO_ID_VJP, [a["q"], a["yd"], np.concatenate([a["aux"], a["w"]], 1)])
    gq, gf = _replay(ctx, g.ALGO_GFS_VJP, [a["q"], a["f"].reshape(len(a["q"]), -1), a["w"]])
    return [idv[0] + gq, idv[1], idv[2], gf]


def _fd_ext_vjp_ref(ctx, a, g):
    ff = a["f"].reshape(len(a["q"]), -1)
    tau_eff = _replay(ctx, g.ALGO_GFA, [a["q"], ff, a["aux"]])[0]
    fdv = _replay(ctx, g.ALGO_FD_VJP, [a["q"], a["yd"], np.concatenate([tau_eff, a["w"]], 1)])
    gq, gf = _replay(ctx, g.ALGO_GFA_VJP, [a["q"], ff, fdv[2]])
    return [fdv[0] + gq, fdv[1], fdv[2], gf]


def entry_points(g):
    o = lambda ctx: ctx["oracle"]  # noqa: E731
    return [
        EntryPoint("contact_kinematics", [g.ALGO_CONTACT_KIN], lambda m, a: m.contactKinematics(a["q"], a["yd"]),
                   lambda c, a: o(c).contact_kinematics(a["q"], a["yd"]), TOL64, "yd"),
        EntryPoint("contact_jacobians", [g.ALGO_CONTACT_JAC], lambda m, a: (m.contactJacobians(a["q"]),),
                   lambda c, a: [o(c).contact_jacobians(a["q"], world=True)], TOL64),
        EntryPoint("apply_test_force", [g.ALGO_TEST_FORCE], lambda m, a: m.applyTestForce(a["q"], a["ft"]),
                   lambda c, a: o(c).apply_test_force(a["q"], a["ft"]), TOL_OSIM, "ft"),
        EntryPoint("inverse_osim", [g.ALGO_OSIM], lambda m, a: (m.inverseOperationalSpaceInertiaMatrix(a["q"]),),
                   lambda c, a: [o(c).inverse_osim(a["q"])], TOL_OSIM),
        EntryPoint("id_jacobians", [g.ALGO_ID_DERIV], lambda m, a: m.inverseDynamicsDerivatives(a["q"], a["yd"], a["aux"]),
                   lambda c, a: o(c).dynamics_derivatives(a["q"], a["yd"], a["aux"], False), TOL64, "yd"),
        EntryPoint("fd_jacobians", [g.ALGO_FD_DERIV], lambda m, a: m.forwardDynamicsDerivatives(a["q"], a["yd"], a["aux"]),
                   lambda c, a: o(c).dynamics_derivatives(a["q"], a["yd"], a["aux"], True), TOL_FD, "aux"),
        EntryPoint("id_vjp", [g.ALGO_ID_VJP], lambda m, a: m.inverseDynamicsVJP(a["q"], a["yd"], a["aux"], a["w"]),
                   lambda c, a: _replay(c, g.ALGO_ID_VJP, [a["q"], a["yd"], np.concatenate([a["aux"], a["w"]], 1)]),
                   TOL64, "yd"),
        EntryPoint("fd_vjp", [g.ALGO_FD_VJP], lambda m, a: m.forwardDynamicsVJP(a["q"], a["yd"], a["aux"], a["w"]),
                   lambda c, a: _replay(c, g.ALGO_FD_VJP, [a["q"], a["yd"], np.concatenate([a["aux"], a["w"]], 1)]),
                   TOL_FD, "yd"),
        EntryPoint("id_vjp_ext", [g.ALGO_ID_VJP, g.ALGO_GFS_VJP],
                   lambda m, a: m.inverseDynamicsVJP(a["q"], a["yd"], a["aux"], a["w"], f_ext=a["f"]),
                   lambda c, a: _id_ext_vjp_ref(c, a, g), TOL64, "yd", extra=1),
        EntryPoint("fd_vjp_ext", [g.ALGO_GFA, g.ALGO_FD_VJP, g.ALGO_GFA_VJP],
                   lambda m, a: m.forwardDynamicsVJP(a["q"], a["yd"], a["aux"], a["w"], f_ext=a["f"]),
                   lambda c, a: _fd_ext_vjp_ref(c, a, g), TOL_FD, "yd", extra=1),
        EntryPoint("contact_vjp", [g.ALGO_CONTACT_KIN_VJP],
                   lambda m, a: m.contactKinematicsVJP(a["q"], a["yd"], a["pb"], a["vb"]),
                   lambda c, a: _replay(c, g.ALGO_CONTACT_KIN_VJP, [a["q"], a["yd"], np.concatenate(
                       [a["pb"].reshape(len(a["q"]), -1), a["vb"].reshape(len(a["q"]), -1)], 1)]), TOL64, "yd"),
        EntryPoint("id_ext", [g.ALGO_ID, g.ALGO_GFS], lambda m, a: (m.inverseDynamics(a["q"], a["yd"], a["aux"], f_ext=a["f"]),),
                   lambda c, a: [o(c).dynamics_with_external_forces(a["q"], a["yd"], a["aux"], a["f"], forward=False)],
                   TOL64, "yd"),
        EntryPoint("fd_ext", [g.ALGO_GFA, g.ALGO_FD], lambda m, a: (m.forwardDynamics(a["q"], a["yd"], a["aux"], f_ext=a["f"]),),
                   lambda c, a: [o(c).dynamics_with_external_forces(a["q"], a["yd"], a["aux"], a["f"], forward=True)],
                   TOL64, "aux"),
    ]


# (model, forced shell): TelloWithArms in the shells its programs select (its derivative programs take minutes to
# compile per shell); the fixed-base chain and a URDF of the corpus in every shell
GPU_CASES = [("tello_with_arms", None)] + [(mod, s) for mod in ("revolute_chain_with_rotor_4", "urdf") for s in SHAPES + [None]]
N_MAX = 3 * 128 + 5
_CTX = {}


def _make_model(grbda, name, device=0):
    if name == "urdf":
        m = grbda.ClusterTreeModel.from_urdf(URDF, device=device)
    else:
        m = grbda.ClusterTreeModel.from_robot(name, device=device)
    # (contact_set places the end-effectors on the force bodies: taken before those become every body)
    m.contacts = contact_set(m)
    m.setContactPoints(*m.contacts)
    m.setExternalForceBodies(list(range(m.nb)))
    return m


def _context(grbda, oracle, torch, name, m, tmp_dir):
    """States, inputs and references of one model, shared by its shells (the programs differ only in their shell)."""
    if name in _CTX:
        return _CTX[name]
    o = oracle.OracleModel(name) if name != "urdf" else mirror_to_oracle(m, oracle)
    o.set_contact_points(*m.contacts)
    q, yd, aux, flags = m.generateStates(N_MAX, seed=13)
    assert int(flags.sum()) == 0
    gen = torch.Generator(device=q.device).manual_seed(21)
    rnd = lambda *shape, s=1.0: (torch.rand(shape, dtype=torch.float64, device=q.device, generator=gen) * 2 - 1) * s  # noqa: E731
    a = dict(q=q, yd=yd, aux=aux, w=rnd(N_MAX, m.nv), f=rnd(N_MAX, m.nb, 6, s=20.0), ft=rnd(N_MAX, m.ncp, 3, s=0.5),
             pb=rnd(N_MAX, m.ncp, 3), vb=rnd(N_MAX, m.ncp, 3))
    tapes = {}

    def tape(algo):
        if algo not in tapes:
            path = str(tmp_dir / ("%s_%d.tape" % (name, algo)))
            m.dump_program(algo, path)
            tapes[algo] = load_tape(path)
        return tapes[algo]

    # revolute coordinates that get the whole turns: TelloWithArms' hip clamp and arm (test_gpu_parity), else the
    # first and last one-coordinate clusters
    cl = m.clusters()
    if name == "tello_with_arms":
        coords = (cl[1]["position_index"], cl[7]["position_index"])
    else:
        ones = [c["position_index"] for c in cl if c["num_positions"] == 1]
        coords = (ones[0], ones[-1])
    ctx = dict(oracle=o, tape=tape, inputs=a, numpy={k: v.cpu().numpy() for k, v in a.items()}, coords=coords, refs={})
    _CTX[name] = ctx
    return ctx


def _np_outs(outs):
    return [t.detach().cpu().numpy() for t in outs]


def _unaligned(torch, t):
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    u = buf[1:].view(t.shape)
    u.copy_(t)
    assert u.data_ptr() % 16 == 8
    return u


def _slice(a, n):
    return {k: v[:n] for k, v in a.items()}


def _check_shell(info, shape):
    if shape == "D":
        assert info["direct"] and not info["tma"] and info["block"] == 128
    elif shape:
        block, ctas = (int(x) for x in shape.split(",")[1:])
        assert info["tma"] and info["block"] == block and info["min_blocks"] == ctas
    assert info["ready"]


@pytest.mark.gpu
@pytest.mark.parametrize("name,shape", GPU_CASES)
def test_run_time_entry_points_on_edges(grbda, oracle, torch, name, shape, tmp_path_factory, monkeypatch):
    if shape:
        monkeypatch.setenv("GRBDA_JIT_SHAPE", shape)
    else:
        monkeypatch.delenv("GRBDA_JIT_SHAPE", raising=False)
    m = _make_model(grbda, name)  # fresh handle: its kernels are built for this shell
    ctx = _context(grbda, oracle, torch, name, m, tmp_path_factory.mktemp("tapes"))
    a, an = ctx["inputs"], ctx["numpy"]
    ran = []
    for ep in entry_points(grbda):
        # the shell chooseShape takes (the programs are compiled on the first call below)
        blocks = {i["block"] for i in (m.kernel_info(algo) for algo in ep.programs) if i["source"] == "jit"}
        try:
            ep.call(m, _slice(a, 1))
        except grbda.GrbdaError as e:
            # a forced shell whose tiles exceed what one CTA may hold cannot be launched for this program
            assert shape and "MaxDynamicSharedMemorySize" in str(e), str(e)
            ran.append("%s/%s: skipped, %s tiles exceed the shared memory of a CTA" % (name, ep.name, shape))
            continue
        infos = [m.kernel_info(algo) for algo in ep.programs]
        jit = [i for i in infos if i["source"] == "jit"]
        for i in jit:
            _check_shell(i, shape)
        assert {i["block"] for i in jit} == blocks
        ran += ["%s/%s/%s b%d %s" % (name, ep.name, grbda.ALGO_NAMES[p] if p < 5 else p, i["block"],
                                    "D" if i["direct"] else "T") for p, i in zip(ep.programs, infos) if i["source"] == "jit"]
        blocks = {i["block"] for i in jit} | ({64, 128} if len(jit) < len(infos) else set())
        b = max(blocks)
        N = 3 * b + 5
        if ep.name not in ctx["refs"]:
            ctx["refs"][ep.name] = [np.asarray(r) for r in ep.ref(ctx, an)]
        ref = [r.reshape(N_MAX, -1) for r in ctx["refs"][ep.name]]

        def check(outs, rows, want, tol, what):
            for k, (g, r) in enumerate(zip(_np_outs(outs), want)):
                assert rel(g.reshape(len(rows), -1), r) < tol, (ep.name, what, k)

        # odd last tiles (and a single state)
        base = None
        for B in (1, 2 * b + 1, 2 * b + 3, N):
            outs = ep.call(m, _slice(a, B))
            check(outs, range(B), [r[:B] for r in ref], ep.tol, "B=%d" % B)
            base = outs
        # flagged tiles: states r0 (tile 0) and r2 (tile 2) beyond the fast sin/cos range
        r0, r2 = 5, 2 * b + 5
        af = _slice(a, N)
        af["q"] = af["q"].clone()
        af["q"][r0, ctx["coords"][0]] += 2.0 * np.pi * TURNS
        af["q"][r2, ctx["coords"][1]] -= 2.0 * np.pi * TURNS
        outs = ep.call(m, af)
        flagged = np.zeros(N, dtype=bool)
        for blk in blocks:
            for r in (r0, r2):
                flagged[(r // blk) * blk:min(N, (r // blk + 1) * blk)] = True
        anf = {k: v[[r0, r2]].copy() for k, v in an.items()}
        anf["q"] = af["q"][[r0, r2]].cpu().numpy()
        ref_f = [np.asarray(r).reshape(2, -1) for r in ep.ref(ctx, anf)]
        for g, r, r_f in zip(_np_outs(outs), ref, ref_f):
            g = g.reshape(N, -1)
            want = r[:N].copy()
            want[[r0, r2]] = r_f
            assert rel(g[flagged], want[flagged]) < ep.tol, (ep.name, "flagged tiles")
        for g, g0 in zip(outs, base):
            assert torch.equal(g[torch.from_numpy(~flagged).to(g.device)], g0[torch.from_numpy(~flagged).to(g.device)]), \
                (ep.name, "unflagged tiles changed")
        # unaligned inputs: q, then the other per-state input
        before = grbda.launch_count()
        ep.call(m, _slice(a, N))
        torch.cuda.synchronize()
        launches_aligned = grbda.launch_count() - before
        for key in ("q", ep.second) if ep.second else ("q",):
            au = _slice(a, N)
            au[key] = _unaligned(torch, au[key])
            before = grbda.launch_count()
            outs = ep.call(m, au)
            torch.cuda.synchronize()
            launches = grbda.launch_count() - before
            if key == "q" and len(jit) == len(infos) and all(i["tma"] for i in jit):
                assert launches == len(ep.programs) + ep.extra, (ep.name, launches)  # one slow launch per program
            elif all(i["direct"] for i in infos):
                assert launches == launches_aligned
            else:
                assert launches <= launches_aligned
            for g, g0 in zip(_np_outs(outs), _np_outs(base)):
                assert rel(g.reshape(N, -1), g0.reshape(N, -1)) < 1e-12, (ep.name, "unaligned " + key)
            check(outs, range(N), [r[:N] for r in ref], ep.tol, "unaligned " + key)
    print("\n".join(ran))


# ---- guard bands -----------------------------------------------------------------------------------------------
SENTINEL = np.array([0x7FF8DEADBEEFCAFE], dtype=np.int64).view(np.float64)[0]  # a NaN no kernel computes


def _guarded(torch, shape, large):
    """A float64 output of `shape` inside a sentinel-filled buffer: at a 32-byte offset when it is a large output
    (kernels/shapes.h shapeLargeOutput: written with whole-sector stores), else at an 8-byte offset."""
    n = int(np.prod(shape))
    front, back = (4 if large else 1), 64
    buf = torch.full((front + n + back,), SENTINEL, dtype=torch.float64, device="cuda")
    out = buf[front:front + n].view(shape)
    assert out.data_ptr() % (32 if large else 16) == (0 if large else 8)
    return buf, out, front, n


def _large(k, n):
    return n > 64 or (k > 0 and n > 16)


def _check_guards(torch, guarded):
    for buf, _, front, n in guarded:
        bits = buf.view(torch.int64).cpu().numpy()
        pattern = np.array([SENTINEL]).view(np.int64)[0]
        assert (bits[:front] == pattern).all() and (bits[front + n:] == pattern).all(), "write outside the output"
        assert not (bits[front:front + n] == pattern).any(), "output element not written"


@pytest.mark.gpu
def test_outputs_inside_guard_bands(grbda, torch):
    """Contact kinematics, FD Jacobians, the FD VJP (with and without forces) and the contact VJP through the C ABI,
    each output in a NaN-filled buffer: after an ordinary call every sentinel outside the output is intact and no
    element inside still holds it; the values equal the Python entry points' to 1e-12."""
    L = grbda.lib()
    m = _make_model(grbda, "urdf")
    B = 2 * 128 + 3
    q, yd, aux, _ = m.generateStates(B, seed=3)
    gen = torch.Generator(device="cuda").manual_seed(4)
    w = torch.rand((B, m.nv), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    f = torch.rand((B, m.nb * 6), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    pb = torch.rand((B, m.ncp * 3), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    vb = torch.rand((B, m.ncp * 3), dtype=torch.float64, device="cuda", generator=gen) - 0.5
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    nq, nv, nc3 = m.nq, m.nv, 3 * m.ncp
    cases = [
        (L.grbda_cuda_contact_kinematics_f64, [q, yd], [nc3, nc3], lambda: m.contactKinematics(q, yd)),
        (L.grbda_cuda_forward_dynamics_derivatives_f64, [q, yd, aux], [nv * nv] * 3,
         lambda: [t.transpose(1, 2) for t in m.forwardDynamicsDerivatives(q, yd, aux)]),
        (L.grbda_cuda_forward_dynamics_vjp_f64, [q, yd, aux, w], [nq, nv, nv], lambda: m.forwardDynamicsVJP(q, yd, aux, w)),
        (L.grbda_cuda_forward_dynamics_ext_vjp_f64, [q, yd, aux, f, w], [nq, nv, nv, 6 * m.nb],
         lambda: m.forwardDynamicsVJP(q, yd, aux, w, f_ext=f)),
        (L.grbda_cuda_contact_kinematics_vjp_f64, [q, yd, pb, vb], [nq, nv], lambda: m.contactKinematicsVJP(q, yd, pb, vb)),
    ]
    for fn, ins, widths, python in cases:
        guarded = [_guarded(torch, (B, n), _large(k, n)) for k, n in enumerate(widths)]
        assert fn(m._h, *[P(t) for t in ins], *[P(g[1]) for g in guarded], B, st) == 0, \
            L.grbda_cuda_last_error_string().decode()
        torch.cuda.synchronize()
        _check_guards(torch, guarded)
        for (_, out, _, _), want in zip(guarded, python()):
            assert rel(out.cpu().numpy(), want.reshape(B, -1).cpu().numpy()) < 1e-12


# ---- FP32 forward kinematics -----------------------------------------------------------------------------------
B32 = 2 * 128 + 3  # last tile of 3 states: odd ring classes, tail threads without a state, the hand-copied tail


@pytest.mark.gpu
@pytest.mark.parametrize("robot", ["tello_with_arms", "mini_cheetah", "mit_humanoid", "revolute_chain_with_rotor_2",
                                   "revolute_chain_with_rotor_16", "revolute_rotor_chain", "jvrc1_humanoid", "urdf"])
def test_forward_kinematics_f32(grbda, oracle, torch, robot):
    """FP32 forward kinematics against the FP64 oracle on float-rounded states (the FP32-built models of
    test_dynamics_parity_f32 and one run-time compiled model), and FP32 ID / H at the same batch on TelloWithArms."""
    if robot == "urdf":
        m = grbda.ClusterTreeModel.from_urdf(URDF)
        o = mirror_to_oracle(m, oracle)
    else:
        m = grbda.ClusterTreeModel.from_robot(robot)
        o = oracle_for(oracle, m, robot)
    q, yd, aux, _ = m.generateStates(B32, seed=8)
    q32, yd32, aux32 = q.float(), yd.float(), aux.float()
    qn, ydn, auxn = (x.double().cpu().numpy() for x in (q32, yd32, aux32))
    p, R, v = m.forwardKinematics(q32, yd32)
    assert m.kernel_info(grbda.ALGO_FK, True)["source"] == ("jit" if robot == "urdf" else "aot")
    po, Ro, vo = o.forward_kinematics(qn, ydn)
    for g, r in ((p, po), (R, Ro), (v, vo)):
        g = g.double().cpu().numpy()
        assert np.isfinite(g).all()
        assert np.abs(g - r).max() / np.abs(r).max() < TOL32
    if robot == "tello_with_arms":
        tau = m.inverseDynamics(q32, yd32, aux32).double().cpu().numpy()
        assert relrows(tau, o.inverse_dynamics(qn, ydn, auxn)) < TOL32
        assert relrows(m.getMassMatrix(q32).double().cpu().numpy(), o.mass_matrix(qn)) < TOL32
