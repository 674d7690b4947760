#!/usr/bin/env python
"""Headline benchmark: forward + inverse dynamics evaluations per second, TelloWithArms
(37 bodies, 15 clusters, nq 33, nv 24), 2^20 independent states per GPU, FP64.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torchrun)
  python bench.py --impl reference ...                     (the CPU path on the box's host cores)

A step = one pass of the hot path over one batch of synthetic states: forwardDynamics
(constraint-embedded ABA) followed by inverseDynamics (cluster RNEA) of the resulting accelerations.
`value` counts fwd+inv PAIRS per second summed over all GPUs, inputs resident in HBM; `e2e` is the
same pass through the host-buffer entry point (pinned host memory -> H2D -> kernels -> D2H).
The batch is sharded by global state index, no collective on the data path; the only collective is the
final timing / checksum gather. --scaling weak (default): 2^20 states per GPU; --scaling strong: 2^20
states in total, 2^20 / N per GPU (SURVEY 8(d)/(e)). Whatever the flag, the line carries both measurements
("weak_scaling" / "strong_scaling"); `value`, `ms_per_step` and `scaling` are those of the selected mode.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fwd+inv dynamics evals/s (Tello, batch 2^20)"
UNIT = "fwd+inv state evaluations/s"
# --dump-outputs writes at most this many bytes: beyond it, a fixed seeded sample of the states (rows)
DUMP_BYTES = 48 << 20


def dump_rows(n, cols):
    """Sorted indices of the rows of [n, cols] float64 outputs that --dump-outputs writes: every row if they fit
    DUMP_BYTES, otherwise the same seeded sample on every run."""
    k = DUMP_BYTES // (8 * cols)
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def dump_outputs(out_dir, arrays):
    """arrays: name -> float64 array (the sampled rows of one output), written as out_dir/<name>.npy."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured"
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], stdout=subprocess.PIPE, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(s) > 3 + i and s[3 + i] == "Active" for s in self.samples)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def cpu_baseline(model_name, seconds_target=12.0, threads=0):
    """The oracle (CPU restatement of the reference path) on the host cores, bounded sample."""
    from oracle import binding
    o = binding.OracleModel(model_name)
    cores = binding.max_threads() if threads <= 0 else threads
    n = 256 * cores
    q, yd, tau = o.generate_states(n)
    t0 = time.perf_counter()
    ydd = o.forward_dynamics(q, yd, tau, threads=cores)
    o.inverse_dynamics(q, yd, ydd, threads=cores)
    dt = time.perf_counter() - t0
    # scale the sample to about seconds_target of CPU work
    n2 = int(max(n, min(1 << 18, n * seconds_target / max(dt, 1e-6))))
    q, yd, tau = o.generate_states(n2)
    t0 = time.perf_counter()
    ydd = o.forward_dynamics(q, yd, tau, threads=cores)
    o.inverse_dynamics(q, yd, ydd, threads=cores)
    dt = time.perf_counter() - t0
    return {"value": n2 / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "%d states, forwardDynamics + inverseDynamics, %d threads, %.1f s" % (n2, cores, dt)}, o


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the host cores. The
    reference itself cannot be built here (Eigen / CasADi / urdfdom absent, DESIGN.md), so this is
    the oracle port, all host threads, a bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import binding
    o = binding.OracleModel(args.model)
    cores = binding.max_threads()
    n = args.ref_states
    q, yd, tau = o.generate_states(n)
    for _ in range(args.warmup):
        o.inverse_dynamics(q[:256], yd[:256], o.forward_dynamics(q[:256], yd[:256], tau[:256]))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ydd = o.forward_dynamics(q, yd, tau, threads=cores)
        tau_back = o.inverse_dynamics(q, yd, ydd, threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        rows = dump_rows(n, 2 * o.nv)
        dump_outputs(args.dump_outputs, {"ydd": ydd[rows], "tau_back": tau_back[rows]})
    value = n * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "%s forwardDynamics+inverseDynamics, %d-state sample per step (CPU)" % (args.model, n),
                       "model": args.model, "batch_per_step": n},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d states x %d steps" % (n, args.steps)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def ncu_traffic(kernel, states):
    """DRAM bytes of one launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed ncu
    --set full capture of this round, scaled to `states`; None when no capture is on file."""
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles")
    for name in ("r2_roofline_traffic.json", "r1_roofline_traffic.json"):  # newest capture on file
        try:
            rec = json.load(open(os.path.join(here, name)))[kernel]
            return rec["dram_bytes_per_launch"] * states / rec["states"]
        except (OSError, KeyError, ValueError):
            continue
    return None


_RESULT_FD = None


def _stdout_for_the_result_only():
    """Libraries write to stdout (NCCL prints its version banner there). The contract is ONE JSON line on
    stdout, so everything else is sent to stderr: fd 1 is pointed at fd 2 and the JSON line is written to a
    saved copy of the real stdout by emit()."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    text = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(text.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, text)


def main():
    _stdout_for_the_result_only()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--model", default="tello_with_arms")
    ap.add_argument("--batch", type=int, default=1 << 20, help="states per GPU")
    ap.add_argument("--ref-states", type=int, default=1 << 14)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--scaling", choices=("weak", "strong"), default="weak",
                    help="weak: --batch states per GPU; strong: --batch states in total, sharded")
    ap.add_argument("--no-extras", action="store_true", help="skip the config-3 leg and the depth sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step (ydd of forwardDynamics, tau_back of inverseDynamics; "
                         "rank 0's shard, a fixed seeded sample of its states beyond %d MB) as DIR/<name>.npy, float64"
                         % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    import generalized_rbda_b200 as grbda
    from generalized_rbda_b200.sharding import gather_summary, shard_range, weak_shard

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    # host placement first: the pinned buffers of the end-to-end leg are allocated later by this thread
    numa = grbda.bind_host_to_device(local_rank)
    m = grbda.ClusterTreeModel.from_robot(args.model, device=local_rank)
    B = args.batch
    # contiguous shard of the global index range, generated on this GPU
    first_index, _ = weak_shard(B, rank)
    q, yd, tau, flags = m.generateStates(B, first_index=first_index)
    ydd = torch.empty_like(tau)
    tau_back = torch.empty_like(tau)
    assert int(flags.sum()) == 0
    # strong scaling: the first 2^20 / N states of the same buffers (states are i.i.d.: any contiguous
    # slice of a shard is as good as the rank's slice of the global batch for timing purposes)
    _, Bs = shard_range(B, rank, world)

    def step():
        m.forwardDynamics(q, yd, tau, out=ydd)
        m.inverseDynamics(q, yd, ydd, out=tau_back)

    def step_strong():
        m.forwardDynamics(q[:Bs], yd[:Bs], tau[:Bs], out=ydd[:Bs])
        m.inverseDynamics(q[:Bs], yd[:Bs], ydd[:Bs], out=tau_back[:Bs])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps bracketed by barrier + synchronize, CUDA events, max over ranks (ms for all K steps)."""
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    primary, other = (step, step_strong) if args.scaling == "weak" else (step_strong, step)
    for _ in range(args.warmup):
        other()
    ms_other = timed(other, args.steps)
    for _ in range(args.warmup):
        primary()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = grbda.launch_count()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        primary()
    e1.record()
    barrier()
    launches = grbda.launch_count() - launches0
    ms = e0.elapsed_time(e1)
    dumped = None
    if args.dump_outputs and rank == 0:
        # copied before anything else runs: these are the buffers the last timed step wrote
        rows = torch.from_numpy(dump_rows(B if primary is step else Bs, 2 * m.nv)).to(dev)
        dumped = {"ydd": ydd.index_select(0, rows).cpu().numpy(),
                  "tau_back": tau_back.index_select(0, rows).cpu().numpy()}
    # The timed region lasts ~20 ms, one nvidia-smi query takes longer than that: the sampler keeps running
    # over an untimed continuation of exactly the same steps (about 0.7 s) so that the clocks / throttle
    # reasons reported are a median over several samples under this load.
    timed_samples = len(sampler.samples)
    extra = int(min(2000, max(args.steps, 0.7 / max(ms * 1e-3 / args.steps, 1e-6))))
    for _ in range(extra):
        primary()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_weak, ms_strong = (ms_max, ms_other) if args.scaling == "weak" else (ms_other, ms_max)
    value_weak = world * B * args.steps / (ms_weak * 1e-3)
    value_strong = B * args.steps / (ms_strong * 1e-3)
    value = value_weak if args.scaling == "weak" else value_strong

    # per-kernel timing of the dominant kernel (FD) and of ID, same stream, CUDA events
    def time_kernel(fn, reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps * 1e-3

    t_fd = time_kernel(lambda: m.forwardDynamics(q, yd, tau, out=ydd), args.steps)
    t_id = time_kernel(lambda: m.inverseDynamics(q, yd, ydd, out=tau_back), args.steps)
    # the other two kernels of the path (HBM-write bound): a quarter of the batch keeps memory modest
    Bk = max(1, B // 4)
    Hbuf = torch.empty((Bk, m.nv, m.nv), dtype=torch.float64, device=dev)
    fk_out = m.forwardKinematics(q[:Bk], yd[:Bk])
    m.getMassMatrix(q[:Bk], out=Hbuf)
    t_h = time_kernel(lambda: m.getMassMatrix(q[:Bk], out=Hbuf), 5)
    t_fk = time_kernel(lambda: m.forwardKinematics(q[:Bk], yd[:Bk], out=fk_out), 5)
    del Hbuf, fk_out
    # dynamics with external forces on the terminal links (SURVEY §8 f2): two launches each
    nf = len(m.externalForceBodies())
    f_ext = (torch.rand((B, nf, 6), dtype=torch.float64, device=dev) - 0.5) * 20.0
    ext_out = torch.empty_like(tau)
    m.forwardDynamics(q, yd, tau, out=ext_out, f_ext=f_ext)
    t_fd_ext = time_kernel(lambda: m.forwardDynamics(q, yd, tau, out=ext_out, f_ext=f_ext), 5)
    t_id_ext = time_kernel(lambda: m.inverseDynamics(q, yd, ydd, out=ext_out, f_ext=f_ext), 5)
    del f_ext, ext_out

    # BASELINE config 3: mit_humanoid forwardDynamics + massMatrix, 2^20 (FD) / 2^18 (H) states in total,
    # sharded over the ranks; BASELINE config 5: depth sweep of the serial rotor chain (rank 0, N = 1 only;
    # depths without ahead-of-time kernels are compiled at run time)
    extras = {}
    if not args.no_extras:
        mh = grbda.ClusterTreeModel.from_robot("mit_humanoid", device=local_rank)
        f3, n3 = shard_range(1 << 20, rank, world)
        q3, yd3, tau3, _ = mh.generateStates(n3, first_index=f3)
        out3 = torch.empty_like(tau3)
        n3h = max(1, n3 // 4)
        H3 = torch.empty((n3h, mh.nv, mh.nv), dtype=torch.float64, device=dev)
        mh.forwardDynamics(q3, yd3, tau3, out=out3), mh.getMassMatrix(q3[:n3h], out=H3)
        ms_fd3 = timed(lambda: mh.forwardDynamics(q3, yd3, tau3, out=out3), 10) / 10
        ms_h3 = timed(lambda: mh.getMassMatrix(q3[:n3h], out=H3), 10) / 10
        extras["mit_humanoid_sharded"] = {
            "states_total_fd": 1 << 20, "states_total_h": world * n3h, "n_gpus": world, "fd_ms": ms_fd3, "h_ms": ms_h3,
            "fd_evals_per_s": (1 << 20) / (ms_fd3 * 1e-3), "h_evals_per_s": world * n3h / (ms_h3 * 1e-3),
            "h_hbm_frac_per_gpu": 8 * (mh.nq + mh.nv * mh.nv) * n3h / (ms_h3 * 1e-3) / 1e9 / load_peaks()[0]["hbm_gbs"]}
        del mh, q3, yd3, tau3, out3, H3
        if world == 1:
            # BASELINE config 2: mini_cheetah, 2^20 states, forward + inverse dynamics on one GPU
            mc2 = grbda.ClusterTreeModel.from_robot("mini_cheetah", device=local_rank)
            q2, yd2, tau2, _ = mc2.generateStates(1 << 20)
            o2 = torch.empty_like(tau2)
            mc2.forwardDynamics(q2, yd2, tau2, out=o2), mc2.inverseDynamics(q2, yd2, tau2, out=o2)
            ms_fd2 = timed(lambda: mc2.forwardDynamics(q2, yd2, tau2, out=o2), 10) / 10
            ms_id2 = timed(lambda: mc2.inverseDynamics(q2, yd2, tau2, out=o2), 10) / 10
            extras["mini_cheetah_fwd_inv"] = {"states": 1 << 20, "fd_ms": ms_fd2, "id_ms": ms_id2,
                                              "pairs_per_s": (1 << 20) / ((ms_fd2 + ms_id2) * 1e-3)}
            del mc2, q2, yd2, tau2, o2
            sweep = []
            for depth in (2, 4, 8, 16, 24):
                mc = grbda.ClusterTreeModel.from_robot("revolute_chain_with_rotor_%d" % depth, device=local_rank)
                nS = 1 << 18
                qc, ydc, tc, _ = mc.generateStates(nS)
                oc = torch.empty_like(tc)
                mc.forwardDynamics(qc, ydc, tc, out=oc), mc.inverseDynamics(qc, ydc, tc, out=oc)
                sweep.append({"depth": depth, "states": nS,
                              "fd_ms": timed(lambda: mc.forwardDynamics(qc, ydc, tc, out=oc), 10) / 10,
                              "id_ms": timed(lambda: mc.inverseDynamics(qc, ydc, tc, out=oc), 10) / 10,
                              "kernels": mc.kernel_info(grbda.ALGO_FD)["source"]})
                del mc
            extras["revolute_chain_with_rotor_depth_sweep"] = sweep

    # parity spot check + checksum gather (the only collective)
    err = float(((tau_back - tau).abs().amax(1) / tau.abs().amax(1)).median())
    # the only collective: per-rank checksum / timing summary
    summary = gather_summary(list(grbda.checksum(ydd)) + [ms], device=dev)
    cs = summary[:, :2].sum(0)

    e2e = None
    if not args.no_e2e:
        qh, ydh, tauh = (x.cpu().pin_memory() for x in (q, yd, tau))
        yddh = torch.empty((B, m.nv), dtype=torch.float64).pin_memory()
        tbh = torch.empty((B, m.nv), dtype=torch.float64).pin_memory()

        def e2e_step():
            m.forward_inverse_host(qh, ydh, tauh, yddh, tbh)
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(2, min(args.steps, 5))
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * B * n_e2e / float(dt.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(B * (m.nq + 2 * m.nv) * 8), "d2h_bytes_per_step": int(2 * B * m.nv * 8),
               "steps": n_e2e, "api": "grbda_cuda_forward_inverse_host_f64 (pinned host buffers, 128k-state "
                                      "chunks pipelined over 3 streams)",
               "host_placement": numa}
        assert torch.equal(yddh, ydd.cpu())

    if rank == 0:
        peaks, peaks_kind = load_peaks()
        fd_prog, id_prog = m.kernel_counts(grbda.ALGO_FD), m.kernel_counts(grbda.ALGO_ID)
        fp64_peak = grbda.measure_fma_peak(local_rank, fp32=False, seconds=0.5)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": "%s forwardDynamics + inverseDynamics, %s, FP64" % (
                               args.model, "%d states per GPU" % B if args.scaling == "weak" else
                               "%d states in total sharded over the GPUs" % B),
                           "model": args.model, "batch_per_gpu": B if args.scaling == "weak" else Bs, "nq": m.nq, "nv": m.nv, "bodies": m.nb,
                           "clusters": m.nc, "l2": "inputs (%.0f MB per step) larger than L2, no flush needed" %
                           (B * (m.nq + 3 * m.nv) * 8 / 1e6), "sharding": "contiguous global-index shards, no NCCL on the data path"},
                "gpu_launches": int(launches),
                "weak_scaling": {"value": value_weak, "states_per_gpu": B, "ms_per_step": ms_weak / args.steps},
                "strong_scaling": {"value": value_strong, "states_total": B, "states_per_gpu": Bs,
                                   "ms_per_step": ms_strong / args.steps},
                "clocks": dict(sampler.summary(), samples_inside_timed_region=timed_samples,
                               note="sampled over the timed steps and an untimed continuation of the same steps"),
                "parity": {"median_rel_err_ID_of_FD": err, "checksum_ydd": [float(cs[0]), float(cs[1])]}}
        if e2e:
            line["e2e"] = e2e
        cpu = None
        if not args.no_cpu_baseline and world >= 1:
            cpu, o = cpu_baseline(args.model)
            line["cpu_baseline"] = cpu
            f_alg_fd = o.count_flops(1)["flops_alg"]
            f_alg_id = o.count_flops(0)["flops_alg"]
        else:
            f_alg_fd, f_alg_id = fd_prog["flops"], id_prog["flops"]
        alg_bytes = (m.nq + 3 * m.nv) * 8
        # roofline of the dominant kernel (forward dynamics). achieved / frac count the operations the
        # kernel EXECUTES (add, sub, mul, div = 1, a fused multiply-add = 2) against the measured FP64 FMA
        # peak. The figure SURVEY 8(d) defines - F_alg, the operations of the reference algorithm counted
        # by the oracle's counting scalar - is reported next to it ("algorithmic"): the kernel runs a
        # cheaper algorithm (CRBA + sparse LTDL, rotors as gyrostats), so that ratio can exceed 1.
        line["roofline"] = {
            "kernel": "forwardDynamics (grbda_batched_kernel_tma<double, Body fd, 128, 2>; program: cluster "
                      "CRBA + RNEA bias + branch-sparse LTDL in one depth-first sweep, rotors as gyrostats, "
                      "long-lived values parked in the shared-memory tile rows)",
            "bound": "fp64", "unit": "TFLOP/s",
            "achieved": fd_prog["flops"] * B / t_fd / 1e12, "peak": fp64_peak / 1e12,
            "frac": (fd_prog["flops"] * B / t_fd) / fp64_peak,
            "peak_source": "measured here: dependent-free DFMA loop (grbda_cuda_measure_fma_peak); "
                           "MEASURED_PEAKS.json has no FP64 entry",
            "flops_per_state_executed": fd_prog["flops"],
            "algorithmic": {"flops_per_state": f_alg_fd, "achieved": f_alg_fd * B / t_fd / 1e12,
                            "frac": (f_alg_fd * B / t_fd) / fp64_peak,
                            "note": "F_alg of SURVEY 8(d): operations of the reference's cluster ABA per state "
                                    "(oracle counting scalar), divided by this kernel's time"},
            "kernel_ms": t_fd * 1e3, "traffic": ncu_traffic("forward_dynamics", B),
            "hbm": {"achieved": alg_bytes * B / t_fd / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": alg_bytes * B / t_fd / 1e9 / peaks["hbm_gbs"], "peak_source": peaks_kind,
                    "bytes_per_state": alg_bytes},
            "inverse_dynamics": {"kernel_ms": t_id * 1e3, "flops_per_state_executed": id_prog["flops"],
                                 "achieved": id_prog["flops"] * B / t_id / 1e12,
                                 "frac": (id_prog["flops"] * B / t_id) / fp64_peak,
                                 "algorithmic": {"flops_per_state": f_alg_id, "achieved": f_alg_id * B / t_id / 1e12,
                                                 "frac": (f_alg_id * B / t_id) / fp64_peak},
                                 "hbm_frac": alg_bytes * B / t_id / 1e9 / peaks["hbm_gbs"]}}
        line["other_kernels"] = {
            "dynamics_with_external_forces": {"states": B, "force_bodies": nf, "forward_ms": t_fd_ext * 1e3,
                                              "inverse_ms": t_id_ext * 1e3},
            "mass_matrix": {"states": Bk, "kernel_ms": t_h * 1e3, "bytes_per_state": 8 * (m.nq + m.nv * m.nv),
                            "hbm_frac": 8 * (m.nq + m.nv * m.nv) * Bk / t_h / 1e9 / peaks["hbm_gbs"]},
            "forward_kinematics": {"states": Bk, "kernel_ms": t_fk * 1e3,
                                   "bytes_per_state": 8 * (m.nq + m.nv + 18 * m.nb),
                                   "hbm_frac": 8 * (m.nq + m.nv + 18 * m.nb) * Bk / t_fk / 1e9 / peaks["hbm_gbs"]}}
        line["other_kernels"].update(extras)
        if dumped:
            dump_outputs(args.dump_outputs, dumped)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
