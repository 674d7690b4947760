"""Kernel times of the rigid-contact entry points (contactForwardDynamics, contactImpulse) at 2^20 states, beside plain
forwardDynamics and the composite torch route a user had before them: getMassMatrix + inverseDynamics(ydd = 0) +
contactJacobians + one batched torch.linalg.solve of the KKT system [H J^T; J 0]. That route leaves out the drift
Jdot yd (no entry point gives it), so its time is a lower bound. The inputs of 2^20 states are larger than the 126 MB
L2 (q alone is 150-280 MB). Contact sets: the four feet of Mini Cheetah; the feet and elbows of TelloWithArms and of
the MIT humanoid (the terminal links), every contact active, damping 0. Each record names the card and its power
limit, read in the same run, and gives the operation counts, launch shape, registers / stack bytes per thread
(cuobjdump -res-usage of the run-time compiled cubin) and the NVRTC time of both programs.
Usage: python tools/contact_timing.py > profiles/r6_contact_dynamics.jsonl"""
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import time

# a fresh kernel cache, removed at exit: the first call of each program measures NVRTC, not the disk cache
WORK = tempfile.TemporaryDirectory(prefix="grbda_contact_timing_")
os.environ.setdefault("GRBDA_CACHE_DIR", os.path.join(WORK.name, "cache"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import generalized_rbda_b200 as grbda  # noqa: E402

ROBOTS = ("mini_cheetah", "mit_humanoid", "tello_with_arms")


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
    info = m.kernel_info(algo)
    rec = {"shape": "%s,%d,%d" % ("T" if info["tma"] else "D" if info["direct"] else "S", info["block"],
                                  info["min_blocks"]), "nvrtc_ms": info["compile_ms"]}
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    path = os.path.join(WORK.name, "program%d.cubin" % algo)
    m.jit_compile(algo, False, None, path)
    usage = re.findall(r"REG:(\d+) STACK:(\d+)", subprocess.run([tool, "-res-usage", path], capture_output=True,
                                                                 text=True).stdout)
    rec["registers"] = max(int(r) for r, _ in usage)
    rec["stack_bytes"] = max(int(st) for _, st in usage)
    return rec


def main():
    assert torch.cuda.is_available(), "contact_timing.py measures on a CUDA device"
    gpu_name, power_limit = card()
    for robot in ROBOTS:
        m = grbda.ClusterTreeModel.from_robot(robot)
        bodies = m.externalForceBodies()
        offsets = np.tile([0.0, 0.0, -0.02], (len(bodies), 1))
        m.setContactPoints(bodies, offsets)
        rec = {"model": robot, "nq": m.nq, "nv": m.nv, "contact_points": m.ncp, "gpu": gpu_name,
               "power_limit": power_limit}
        rec.update({k + "_flops": m.dump_program(a)["flops"] for k, a in (
            ("contact_fd", grbda.ALGO_CONTACT_FD), ("contact_impulse", grbda.ALGO_CONTACT_IMPULSE),
            ("fd_ltl", grbda.PROGRAM_FD_LTL))})
        q, yd, tau, _ = m.generateStates(128)
        for name, fn in (("contact_fd", lambda: m.contactForwardDynamics(q, yd, tau)),
                         ("contact_impulse", lambda: m.contactImpulse(q, yd))):
            t0 = time.time()
            fn()
            torch.cuda.synchronize()
            rec[name + "_first_call_s"] = round(time.time() - t0, 2)
        for name, algo in (("contact_fd", grbda.ALGO_CONTACT_FD), ("contact_impulse", grbda.ALGO_CONTACT_IMPULSE)):
            rec.update({name + "_" + k: v for k, v in resources(m, algo).items()})
        B = 1 << 20
        rec["states"] = B
        q, yd, tau, flags = m.generateStates(B)
        rec["flagged_states"] = int(flags.sum())
        out = torch.empty_like(tau)
        rec["fd_ms"] = round(timeit(lambda: m.forwardDynamics(q, yd, tau, out=out)), 4)
        rec["contact_fd_ms"] = round(timeit(lambda: m.contactForwardDynamics(q, yd, tau)), 4)
        rec["contact_impulse_ms"] = round(timeit(lambda: m.contactImpulse(q, yd, restitution=0.2)), 4)
        nv, mm = m.nv, 3 * m.ncp
        zero = torch.zeros_like(tau)

        def composite():
            H = m.getMassMatrix(q)
            C = m.inverseDynamics(q, yd, zero)
            J = m.contactJacobians(q)[:, :, 3:, :].reshape(B, mm, nv)
            K = torch.zeros(B, nv + mm, nv + mm, dtype=torch.float64, device=q.device)
            K[:, :nv, :nv] = H
            K[:, :nv, nv:] = J.transpose(1, 2)
            K[:, nv:, :nv] = J
            rhs = torch.zeros(B, nv + mm, dtype=torch.float64, device=q.device)
            rhs[:, :nv] = tau - C
            return torch.linalg.solve(K, rhs)

        rec["composite_torch_route_ms"] = round(timeit(composite, reps=3), 4)
        rec["composite_torch_route_note"] = "drift Jdot yd omitted: lower bound"
        rec["contact_fd_speedup_vs_composite"] = round(rec["composite_torch_route_ms"] / rec["contact_fd_ms"], 2)
        print(json.dumps(rec), flush=True)
        del q, yd, tau, out, zero
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
    WORK.cleanup()
