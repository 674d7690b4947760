"""Kernel times of the vector-Jacobian product programs (reverse mode) and, beside them, the Jacobian route they
replace: the Jacobian entry point followed by torch.bmm of the cotangent with each matrix. The Jacobian route of the
inverse dynamics is timed without H w (it would need the mass-matrix kernel and one more bmm): its time is a lower
bound. Each record names the card and its power limit, read in the same run, and gives the operation counts of the
programs and, for the VJP kernels, the launch shape and the registers / stack (local memory) per thread that
cuobjdump -res-usage reports for the cubin (the largest over the kernels of the cubin).

--ext-contact: the vector-Jacobian products with external forces and of the contact kinematics instead, 2^20 states of
TelloWithArms (default force bodies), Mini Cheetah and MIT humanoid with the contact set of the tests: the forward
entry points, their VJPs, and for the contact kinematics the route contactJacobians + einsum (yd_bar = J_lin^T v_bar
only) at the largest batch of 2^20, 2^19, ... whose J fits in half the free memory. No Jacobian entry point takes
external forces, so the dynamics with forces have no Jacobian route.
Usage: python tools/vjp_timing.py > profiles/r3_vjp.jsonl
       python tools/vjp_timing.py --ext-contact > profiles/r4_ext_contact_vjp.jsonl"""
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

# a fresh kernel cache, removed at exit: the first call of each program measures NVRTC, not the disk cache
WORK = tempfile.TemporaryDirectory(prefix="grbda_vjp_timing_")
os.environ.setdefault("GRBDA_CACHE_DIR", os.path.join(WORK.name, "cache"))

import torch  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import generalized_rbda_b200 as grbda  # noqa: E402

ROBOTS = ("revolute_chain_with_rotor_8", "mini_cheetah", "mit_humanoid", "tello_with_arms")
LOG2_BATCHES = (16, 20)


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    name, power = [s.strip() for s in out.split(",")]
    return name, power


def resources(m, algo):
    """Launch shape, and registers / stack bytes per thread of the run-time compiled cubin of one program."""
    info = m.kernel_info(algo)
    rec = {"shape": "%s,%d,%d" % ("T" if info["tma"] else "D" if info["direct"] else "S", info["block"],
                                  info["min_blocks"])}
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if os.path.exists(tool):
        path = os.path.join(WORK.name, "program%d.cubin" % algo)
        m.jit_compile(algo, False, None, path)
        usage = re.findall(r"REG:(\d+) STACK:(\d+)", subprocess.run([tool, "-res-usage", path], capture_output=True,
                                                                     text=True).stdout)
        if usage:
            rec["registers"] = max(int(r) for r, _ in usage)
            rec["stack_bytes"] = max(int(st) for _, st in usage)
    return rec


def first_call(fn):
    t0 = time.time()
    fn()
    torch.cuda.synchronize()
    return round(time.time() - t0, 2)


def ext_contact(gpu_name, power_limit):
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    from test_compiler_cpu import contact_set
    for robot in ("tello_with_arms", "mini_cheetah", "mit_humanoid"):
        m = grbda.ClusterTreeModel.from_robot(robot)
        bodies, offsets, ee = contact_set(m)
        m.setContactPoints(bodies, offsets, ee)
        nf = len(m.externalForceBodies())
        rec = {"model": robot, "nq": m.nq, "nv": m.nv, "force_bodies": nf, "contact_points": m.ncp,
               "gpu": gpu_name, "power_limit": power_limit}
        rec.update({k + "_flops": m.dump_program(a)["flops"] for k, a in (
            ("gfa", grbda.ALGO_GFA), ("gfs", grbda.ALGO_GFS), ("gfa_vjp", grbda.ALGO_GFA_VJP),
            ("gfs_vjp", grbda.ALGO_GFS_VJP), ("contact_kin", grbda.ALGO_CONTACT_KIN),
            ("contact_jac", grbda.ALGO_CONTACT_JAC), ("contact_kin_vjp", grbda.ALGO_CONTACT_KIN_VJP))})
        q, yd, aux, _ = m.generateStates(128)
        w, f = torch.rand_like(aux), torch.rand(128, nf, 6, dtype=torch.float64, device=q.device)
        rec["id_ext_vjp_first_call_s"] = first_call(lambda: m.inverseDynamicsVJP(q, yd, aux, w, f_ext=f))
        rec["fd_ext_vjp_first_call_s"] = first_call(lambda: m.forwardDynamicsVJP(q, yd, aux, w, f_ext=f))
        p_bar = torch.rand(128, m.ncp, 3, dtype=torch.float64, device=q.device)
        rec["contact_kin_vjp_first_call_s"] = first_call(lambda: m.contactKinematicsVJP(q, yd, p_bar, p_bar))
        for name, algo in (("gfa_vjp", grbda.ALGO_GFA_VJP), ("gfs_vjp", grbda.ALGO_GFS_VJP),
                           ("contact_kin_vjp", grbda.ALGO_CONTACT_KIN_VJP)):
            rec[name + "_nvrtc_ms"] = m.kernel_info(algo)["compile_ms"]
            rec.update({name + "_" + k: v for k, v in resources(m, algo).items()})
        B = 1 << 20
        rec["states"] = B
        q, yd, aux, _ = m.generateStates(B)
        w = torch.rand_like(aux) * 2 - 1
        f = torch.rand(B, nf, 6, dtype=torch.float64, device=q.device) * 40 - 20
        out = torch.empty_like(aux)
        rec["id_ext_ms"] = round(timeit(lambda: m.inverseDynamics(q, yd, aux, out=out, f_ext=f)), 4)
        rec["fd_ext_ms"] = round(timeit(lambda: m.forwardDynamics(q, yd, aux, out=out, f_ext=f)), 4)
        rec["id_ext_vjp_ms"] = round(timeit(lambda: m.inverseDynamicsVJP(q, yd, aux, w, f_ext=f)), 4)
        rec["fd_ext_vjp_ms"] = round(timeit(lambda: m.forwardDynamicsVJP(q, yd, aux, w, f_ext=f)), 4)
        rec["id_vjp_ms"] = round(timeit(lambda: m.inverseDynamicsVJP(q, yd, aux, w)), 4)
        rec["fd_vjp_ms"] = round(timeit(lambda: m.forwardDynamicsVJP(q, yd, aux, w)), 4)
        del aux, w, f, out
        p_bar = torch.rand(B, m.ncp, 3, dtype=torch.float64, device=q.device) * 2 - 1
        v_bar = torch.rand_like(p_bar) * 2 - 1
        rec["contact_kin_ms"] = round(timeit(lambda: m.contactKinematics(q, yd)), 4)
        rec["contact_kin_vjp_ms"] = round(timeit(lambda: m.contactKinematicsVJP(q, yd, p_bar, v_bar)), 4)
        Bj = B
        while Bj * m.ncp * 6 * m.nv * 8 > torch.cuda.mem_get_info()[0] // 2:
            Bj //= 2
        qj, vj = q[:Bj], v_bar[:Bj]
        rec["contact_jacobian_route_states"] = Bj
        rec["contact_jacobian_route_ms"] = round(timeit(
            lambda: torch.einsum("bci,bcik->bk", vj, m.contactJacobians(qj)[:, :, 3:, :])), 4)
        rec["contact_kin_vjp_ms_at_route_states"] = round(timeit(
            lambda: m.contactKinematicsVJP(qj, yd[:Bj], p_bar[:Bj], vj)), 4)
        print(json.dumps(rec), flush=True)
        del q, yd, p_bar, v_bar, qj, vj
        torch.cuda.empty_cache()


gpu_name, power_limit = card()
if "--ext-contact" in sys.argv:
    ext_contact(gpu_name, power_limit)
    WORK.cleanup()
    sys.exit(0)
for robot in ROBOTS:
    m = grbda.ClusterTreeModel.from_robot(robot)
    flops = {k: m.dump_program(a)["flops"] for k, a in (("id", grbda.ALGO_ID), ("fd_ltl", grbda.PROGRAM_FD_LTL),
                                                         ("id_vjp", grbda.ALGO_ID_VJP), ("fd_vjp", grbda.ALGO_FD_VJP),
                                                         ("id_deriv", grbda.ALGO_ID_DERIV),
                                                         ("fd_deriv", grbda.ALGO_FD_DERIV))}
    q, yd, aux, _ = m.generateStates(128)
    w = torch.rand_like(aux)
    first = {"id_vjp_first_call_s": first_call(lambda: m.inverseDynamicsVJP(q, yd, aux, w)),
             "fd_vjp_first_call_s": first_call(lambda: m.forwardDynamicsVJP(q, yd, aux, w)),
             "id_vjp_nvrtc_ms": m.kernel_info(grbda.ALGO_ID_VJP)["compile_ms"],
             "fd_vjp_nvrtc_ms": m.kernel_info(grbda.ALGO_FD_VJP)["compile_ms"]}
    for name, algo in (("id_vjp", grbda.ALGO_ID_VJP), ("fd_vjp", grbda.ALGO_FD_VJP)):
        first.update({name + "_" + k: v for k, v in resources(m, algo).items()})
    for log2 in LOG2_BATCHES:
        B = 1 << log2
        q, yd, aux, _ = m.generateStates(B)
        w = torch.rand_like(aux) * 2 - 1
        out = torch.empty_like(aux)
        wr = w.unsqueeze(1)

        def id_jacobian_route():
            dq, dv = m.inverseDynamicsDerivatives(q, yd, aux)
            return torch.bmm(wr, dq), torch.bmm(wr, dv)

        def fd_jacobian_route():
            dq, dv, dt = m.forwardDynamicsDerivatives(q, yd, aux)
            return torch.bmm(wr, dq), torch.bmm(wr, dv), torch.bmm(wr, dt)

        rec = {"model": robot, "nq": m.nq, "nv": m.nv, "states": B, "gpu": gpu_name, "power_limit": power_limit}
        rec["id_ms"] = round(timeit(lambda: m.inverseDynamics(q, yd, aux, out=out)), 4)
        rec["fd_ms"] = round(timeit(lambda: m.forwardDynamics(q, yd, aux, out=out)), 4)
        rec["id_vjp_ms"] = round(timeit(lambda: m.inverseDynamicsVJP(q, yd, aux, w)), 4)
        rec["fd_vjp_ms"] = round(timeit(lambda: m.forwardDynamicsVJP(q, yd, aux, w)), 4)
        rec["id_jacobian_route_ms"] = round(timeit(id_jacobian_route), 4)
        rec["fd_jacobian_route_ms"] = round(timeit(fd_jacobian_route), 4)
        rec["id_vjp_speedup_vs_jacobian_route"] = round(rec["id_jacobian_route_ms"] / rec["id_vjp_ms"], 2)
        rec["fd_vjp_speedup_vs_jacobian_route"] = round(rec["fd_jacobian_route_ms"] / rec["fd_vjp_ms"], 2)
        rec.update({k + "_flops": v for k, v in flops.items()})
        rec.update(first)
        print(json.dumps(rec), flush=True)
        del q, yd, aux, w, out, wr
        torch.cuda.empty_cache()
WORK.cleanup()
