#!/usr/bin/env python
"""bench.py -- OCP-QP solves/sec (fp64, batched) of the cuipm CUDA path on chain-mass nx=21 nu=3 N=40.

Contract (see the task brief): ``python bench.py --gpus N --steps K --warmup W`` prints ONE JSON line on rank 0.
A "step" is one pass of the hot path (the whole interior-point solve, one kernel launch) over one batch of
synthetic QPs.  Per-GPU work is fixed (``--batch`` QPs per GPU, default 4096 = BASELINE.json configs[1]), so N>1
is weak scaling; ranks are independent (the batch is the only sharding axis, no data-path collective).

  value        whole-job QP solves/s with the QP records already resident in HBM, timed with CUDA events on the
               solver's stream, max over ranks.
  e2e          the same metric through the C-ABI host entry (cuipm_solve_host_async / cuipm_wait, what
               cuipm_solve_host is made of): pinned HOST buffers, H2D of the QP records and D2H of the solutions and
               per-QP info of every step inside the timed region; two solver objects alternate so that the copies of
               one step overlap the solve of the previous one.
  roofline     HBM roofline of the solve kernel on algorithmic bytes (DESIGN.md section 5).
  cpu_baseline the unmodified reference (HPIPM+BLASFEO behind acados' qp_solver vtable, oracle/_ref) on the host
               cores, bounded sample of the same workload.  ``--impl reference`` times only that arm.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "OCP-QP solves/sec (fp64, batch) chain-mass N=40"
UNIT = "QP/s"


# BASELINE.json configs: (metric suffix, default batch per GPU, description).  c2 is the configuration the metric is quoted on and
# the default; the others are the parity-test shapes, measurable with --config for the per-shape lines of DESIGN.md section 5b.
CONFIGS = {
    "c2": ("chain-mass N=40", 4096, "chain-of-masses OCP-QP nx=21 nu=3 N=40 (after x0 elimination), nbu=3 hard + 4 one-sided soft state bounds (ns=4)"),
    "c1": ("mass-spring N=15", 16384, "mass_spring_example OCP-QP nx=8 nu=3 N=15 (after x0 elimination), input and state boxes"),
    "c3": ("pendulum-sized N=20", 16384, "pendulum-on-cart sized OCP-QP nx=4 nu=1 N=20, input box"),
    "c4": ("quadrotor-sized N=50", 8192, "quadrotor sized OCP-QP nx=12 nu=4 N=50 (uncondensed), input boxes + 6 soft state bounds"),
    "c5": ("legged-sized N=30", 1024, "legged-robot sized OCP-QP nx=48 nu=12 N=30, input boxes + 12 soft state bounds"),
}
_CONFIG = "c2"


def workload(batch: int, seed: int):
    from acados_b200 import problems
    if _CONFIG == "c2":
        return problems.chain_mass(batch, n_mass=5, N=40, seed=seed)
    return problems.named_config(_CONFIG, batch, seed=seed)


def algorithmic_bytes_per_qp(b) -> dict:
    """B_min = 8(|qp_in|+|qp_out|): every QP record is read at least once and its solution written once.
    B_stream = per-iteration streaming model of SURVEY.md 8(d): qp_in + L written + 3 sweeps reading L and BAt."""
    lay, sh = b.layout, b.shape
    qp_in = sum(lay.size[f][k] for f in ("BAt", "RSQ", "DCt", "b", "rq", "d", "dmask", "Z", "z") for k in range(sh.N + 1))
    qp_out = sum(lay.size[f][k] for f in ("ux", "pi", "lam", "t") for k in range(sh.N + 1))
    L = sum(sh.nv(k) ** 2 for k in range(sh.N + 1))
    BA = sum(lay.size["BAt"][k] for k in range(sh.N + 1))
    return {"B_min": 8 * (qp_in + qp_out), "B_stream_iter": 8 * (qp_in + L + 3 * (L + BA))}


def flops_per_qp(b, iters: float) -> float:
    """F_QP = F_res + I * (F_fact + 2 F_solve + 2 F_res), SURVEY.md 8(d)."""
    sh = b.shape
    F_fact = F_solve = F_res = 0.0
    for k in range(sh.N + 1):
        nx, nu, n = sh.nx[k], sh.nu[k], sh.nv(k)
        nx1 = sh.nx_next(k)
        F_fact += 2 * (n + 1) * nx1 * nx1 / 2 + (n + 1) * n * nx1 + n ** 3 / 3.0 + 2 * sh.ng[k] * n * n
        F_solve += 4 * n * nx1 + 2 * n * n + 4 * nx1 * nx1
        F_res += 2 * n * n + 4 * n * nx1
    return F_res + iters * (F_fact + 2 * F_solve + 2 * F_res)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML polled every 10 ms by a thread (the timed region of
    the default run lasts a fraction of a second, shorter than the start-up of an nvidia-smi process); the same fields as the
    nvidia-smi line of the profiling recipe (clocks.sm, clocks.max.sm, clocks_event_reasons.*)."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        self.index, self.samples, self.thread, self.stop_flag, self.h, self.err = index, [], None, False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                phys = int(vis.split(",")[index])
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.smmax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001
            self.err = f"NVML unavailable: {e}"

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, rs))
            except Exception as e:  # noqa: BLE001
                self.err = str(e)
                break
            time.sleep(0.01)

    def start(self):
        if self.h is None:
            return
        self.samples, self.stop_flag = [], False
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def stop(self) -> dict:
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "NVML unavailable"], "samples": 0}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        sm = [m for m, _ in self.samples]
        reasons = sorted({name for _, r in self.samples for name, bit in self.REASONS if r & bit})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.smmax, "reasons": reasons, "samples": len(sm),
                "source": "NVML, 10 ms period, timed region only"}


DUMP_BYTES = 60_000_000


def dump_outputs(dirname: str, b, sol: np.ndarray, info: np.ndarray):
    """What the timed path returned in its last step, as float64 .npy files under DUMP_BYTES in all: the per-QP info fields
    and input trajectories of every QP, and the whole solution records of a fixed, seeded sample of QPs (sorted rows in
    sol_rows.npy).  When even the per-QP arrays of every QP do not fit, they are taken on one seeded sample of rows too
    (qp_rows.npy), of which the solution records are a subset."""
    os.makedirs(dirname, exist_ok=True)
    nb = b.nbatch
    out = {f: info[f].astype(np.float64) for f in ("status", "iter", "res_max", "mu", "obj", "dual_gap", "lq_count")}
    out["u"] = b.layout.u_traj(sol)
    rng = np.random.default_rng(0)
    row_bytes = sum(a.nbytes for a in out.values()) // nb + 8
    if row_bytes * nb > DUMP_BYTES // 2:
        qp_rows = np.sort(rng.choice(nb, DUMP_BYTES // 2 // row_bytes, replace=False))
        out = {name: a[qp_rows] for name, a in out.items()}
        out["qp_rows"] = qp_rows.astype(np.float64)
    else:
        qp_rows = np.arange(nb)
    room = DUMP_BYTES - sum(a.nbytes for a in out.values())
    k = min(len(qp_rows), room // (8 * (b.layout.sol_stride + 1)))
    rows = np.sort(rng.choice(qp_rows, k, replace=False))
    out["sol_rows"], out["sol"] = rows.astype(np.float64), np.ascontiguousarray(sol[rows])
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def cpu_reference(batch_obj, opts, nqp: int, threads: int = 0):
    """Times the unmodified reference on the host cores on the first nqp QPs of the workload."""
    from acados_b200.problems import Batch
    from oracle import oracle_binding as ob
    sub = Batch(batch_obj.shape, batch_obj.layout, np.ascontiguousarray(batch_obj.qp[:nqp]), batch_obj.name)
    if threads <= 0:   # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1: do not rely on the OpenMP default)
        from acados_b200.binding import host_threads
        threads = host_threads()   # affinity mask capped by the cgroup CPU quota: more threads than that only burn the quota
    if ob.have_ref():
        ob.ref_solve(Batch(sub.shape, sub.layout, sub.qp[:min(nqp, 64)].copy()), opts, nthreads=threads)  # warm-up
        sol, info, tm = ob.ref_solve(sub, opts, nthreads=threads)
        # time inside the reference's own evaluate() only (max over threads): its inputs are already in its own
        # panel-major structs, the conversion from cuipm records done by the harness is not charged to the reference
        kind, secs, cores, wall = "reference", tm["solve_s"], tm["threads"], tm["wall_s"]
    else:   # oracle port (only when oracle/_ref could not be built)
        t0 = time.perf_counter()
        sol, info = ob.oracle_solve(sub, opts, nthreads=threads)
        secs, kind, cores = time.perf_counter() - t0, "port", threads or os.cpu_count()
        wall = secs
    return {"value": nqp / secs, "unit": UNIT, "cores": int(cores), "kind": kind,
            "sample": f"{nqp} QPs of the workload, one solver object per OpenMP thread (the structure of the reference's batch "
                      f"solver), time inside ocp_qp_hpipm() only, max over threads; mean IPM iterations {float(info['iter'].mean()):.2f}",
            "value_incl_struct_packing": nqp / wall}, sol, info


def main():
    # the contract is ONE line on stdout: keep the real stdout aside and send everything else that writes to file descriptor 1
    # (NCCL prints its version banner there when a communicator is created) to stderr
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuipm", choices=["cuipm", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="QPs per GPU (default: the configuration's, 4096 for c2)")
    ap.add_argument("--warps", type=int, default=0, help="warps per QP (0 = solver default)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="QPs in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--fast", type=int, default=1, help="0: keep the throughput kernel off (generic one-warp-per-QP kernel only)")
    ap.add_argument("--target-batch", type=int, default=0, help="QPs per GPU of the extra target-point measurement (default: 8192 when the job has 8 ranks)")
    ap.add_argument("--e2e-pipe", type=int, default=1, help="chunks per host call in the e2e leg (0: the solver's default of 8, best for one blocking call; "
                    "1: the whole batch per call, best when two solver objects alternate -- measured 107 k vs 88 k QP/s)")
    ap.add_argument("--no-scatter", action="store_true", help="N > 1: skip the scatter / solve / gather leg over NCCL")
    ap.add_argument("--no-plugin", action="store_true", help="skip the end-to-end leg through the plugin's batched entry")
    ap.add_argument("--no-tight", action="store_true", help="skip the second parity pass (all tolerances 1e-12)")
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS), help="BASELINE.json configuration (default c2: the one the metric is quoted on)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="", help="write what the timed path returned in its last step to DIR/<name>.npy "
                    "(float64, at most 60 MB; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global _CONFIG, METRIC
    _CONFIG = args.config
    if args.batch <= 0:
        args.batch = CONFIGS[_CONFIG][1]
    METRIC = "OCP-QP solves/sec (fp64, batch) " + CONFIGS[_CONFIG][0]

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    steps, warmup = args.steps, max(args.warmup, 0)

    from acados_b200.binding import INFO_DTYPE, default_opts, host_threads
    opts = default_opts()   # what PARTIAL_CONDENSING_HPIPM runs with out of the box
    config = {"workload": f"{CONFIGS[_CONFIG][2]}, batch={args.batch} per GPU, every QP its own matrices", "name": _CONFIG,
              "batch_per_gpu": args.batch, "global_batch": args.batch * max(world, 1), "parallelism": f"batch-sharded x{max(world,1)}",
              "solver_opts": "acados defaults: BALANCE mode, iter_max=50, tol 1e-6/1e-8/1e-8/1e-8, mu0=1, cold start",
              "l2": "inputs (hundreds of MB to GB per batch) exceed the 126 MB L2; no explicit flush"}

    # ------------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        sample = args.cpu_sample or args.batch
        b = workload(sample, seed=1234)
        solve_s, wall_s = [], []
        for it in range(warmup + steps):
            base, rsol, info = cpu_reference(b, opts, sample)
            if it >= warmup:
                # cpu_reference runs a 64-QP warm-up + the sample; use its own clocks of the sample
                solve_s.append(sample / base["value"])
                wall_s.append(sample / base["value_incl_struct_packing"])
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, b, rsol, info)
        val = sample * steps / sum(solve_s)
        base["value"], base["value_incl_struct_packing"] = val, sample * steps / sum(wall_s)
        line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
                "ms_per_step": 1e3 * sample / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": base, "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        real_stdout.write(json.dumps(line) + "\n"); real_stdout.flush()
        return 0

    # ------------------------------------------------------------------------------------------------
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the cuipm path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from acados_b200.binding import CuipmSolver
    b = workload(args.batch, seed=1234 + rank)
    nb = b.nbatch
    solver = CuipmSolver(b.shape, nb, device=local_rank)
    if args.warps:
        solver.set_tuning("warps", args.warps)
    solver.set_tuning("fast", args.fast)
    stream = torch.cuda.ExternalStream(solver.lib.cuipm_stream(solver.handle), device=torch.device("cuda", local_rank))

    # pinned host buffers (the plugin's view) and device-resident copies (the kernel-only view)
    h_qp = torch.from_numpy(b.qp).pin_memory()
    h_sol = torch.zeros((nb, b.layout.sol_stride), dtype=torch.float64).pin_memory()
    h_info = torch.zeros(nb * INFO_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    d_qp = h_qp.cuda()
    d_sol = torch.zeros((nb, b.layout.sol_stride), dtype=torch.float64, device="cuda")
    d_info = torch.zeros(nb * INFO_DTYPE.itemsize, dtype=torch.uint8, device="cuda")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        solver.solve_device(nb, d_qp.data_ptr(), d_sol.data_ptr(), d_info.data_ptr(), opts, sync=False)

    # ---- kernel-only: inputs resident in HBM
    for _ in range(warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record()
    kernel_ms = []
    for _ in range(steps):
        step_device()
    with torch.cuda.stream(stream):
        ev1.record()
    barrier()
    launches_per_step = solver.last_launch_count
    clocks = sampler.stop()
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, b, d_sol.cpu().numpy(), np.frombuffer(d_info.cpu().numpy().tobytes(), dtype=INFO_DTYPE))
    # per-launch duration of the solve kernel (events recorded around each launch by the solver itself)
    solver.solve_device(nb, d_qp.data_ptr(), d_sol.data_ptr(), d_info.data_ptr(), opts, sync=True)
    solve_ms = solver.last_kernel_ms                 # all kernels of one solve (repack, throughput kernel, generic kernel over hand-backs)
    kernel_ms = solver.last_main_kernel_ms           # the dominant kernel alone (CUDA events around its launch on the solver's stream)
    handed_back = solver.last_handed_back
    info = np.frombuffer(d_info.cpu().numpy().tobytes(), dtype=INFO_DTYPE)
    iters_mean = float(info["iter"].mean())

    # ---- end to end through the C-ABI host entry: every step copies its inputs from pinned host memory and its
    # solutions + per-QP info back.  Two solver objects are used alternately through the asynchronous form of the entry
    # (cuipm_solve_host_async / cuipm_wait), so that the transfers of one step overlap the solve of the previous one --
    # the double buffering any streaming caller would use; nothing is skipped, all copies are inside the timed region.
    solver2 = CuipmSolver(b.shape, nb, device=local_rank)
    if args.warps:
        solver2.set_tuning("warps", args.warps)
    solver2.set_tuning("fast", args.fast)
    if args.e2e_pipe:
        solver.set_tuning("pipe", args.e2e_pipe)
        solver2.set_tuning("pipe", args.e2e_pipe)
    h_sol2 = torch.zeros((nb, b.layout.sol_stride), dtype=torch.float64).pin_memory()
    h_info2 = torch.zeros(nb * INFO_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
    lanes = [(solver, h_sol, h_info), (solver2, h_sol2, h_info2)]

    def submit(i):
        sv, hs, hi = lanes[i % 2]
        sv.wait()
        sv.solve_host_async(nb, h_qp.data_ptr(), hs.data_ptr(), hi.data_ptr(), opts)

    def drain():
        for sv, _, _ in lanes:
            sv.wait()

    for i in range(max(2, min(warmup, 4))):
        submit(i)
    drain()
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        submit(i)
    drain()
    barrier()
    e2e_s = time.perf_counter() - t0
    assert np.array_equal(h_info.numpy(), h_info2.numpy()) or steps < 2, "the two lanes solved the same batch: results must agree"
    hinfo = np.frombuffer(h_info.numpy().tobytes(), dtype=INFO_DTYPE)

    # ---- end to end through the PLUGIN: n panel-major ocp_qp_in objects (the reference's structs, built once, untimed) handed to
    # ocp_qp_cuipm_batch_solve of the patched libacados (integration/): per call, inside the timed region, the structs are
    # unpacked into page-locked records by the host threads, copied to the device, solved, copied back and packed into
    # ocp_qp_out objects -- the call a user of PARTIAL_CONDENSING_CUIPM makes.  Single process, N=1 only.
    plugin = None
    if world == 1 and not args.no_plugin:
        try:
            from integration import plugin_bench as pb
            if pb.available():
                pbatch = pb.PluginBatch(b, opts)
                pst, psec = pbatch.run(2 + steps)
                psol, pit, pstat = pbatch.solutions()
                pbatch.close()
                psec = psec[2:]
                plugin = {"value": nb / float(psec.mean()), "unit": UNIT, "ms_per_call": 1e3 * float(psec.mean()), "calls": int(steps),
                          "entry": "ocp_qp_cuipm_batch_solve(config, n, ocp_qp_in**, ocp_qp_out**, opts, mem, status) -- acados_b200/plugin/ocp_qp_cuipm.c",
                          "worst_acados_status": int(pst), "host_threads": host_threads(),
                          "max_abs_dsol_vs_record_path": float(np.max(np.abs(psol - h_sol.numpy()))),
                          "iter_equal_record_path": bool(np.array_equal(pit, hinfo["iter"]))}
            else:
                plugin = {"value": None, "unavailable": "integration/_build/libplugin_bench.so not built (needs the reference sources at build time)"}
        except Exception as e:  # noqa: BLE001
            plugin = {"value": None, "unavailable": str(e)}

    # ---- N > 1: the north_star's data path -- rank 0 holds the records of the WHOLE batch on its device, scatters the shards over
    # NCCL (NVLink), every rank solves its shard, the solutions are gathered on rank 0.  Scatter, solve and gather are all inside
    # the timed region (CUDA events on the current stream, which the NCCL operations are ordered with; max over ranks).
    sg = None
    if world > 1 and not args.no_scatter:
        from acados_b200.sharding import gather_records, scatter_records
        full = d_qp.repeat(world, 1) if rank == 0 else None          # world x batch records on rank 0 (copies of its own batch)
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        seg = np.zeros((0, 3))
        for it in range(1 + min(steps, 3)):
            barrier()
            evs[0].record()
            mine = scatter_records(full)
            evs[1].record()
            torch.cuda.current_stream().synchronize()
            solver.solve_device(nb, mine.data_ptr(), d_sol.data_ptr(), d_info.data_ptr(), opts, sync=True)
            evs[2].record()
            allsol = gather_records(d_sol, nb * world)
            evs[3].record()
            torch.cuda.synchronize()
            if it > 0:     # first pass: NCCL channel set-up
                seg = np.vstack([seg, [evs[0].elapsed_time(evs[1]), evs[1].elapsed_time(evs[2]), evs[2].elapsed_time(evs[3])]])
            del mine
        tt = torch.tensor(seg.mean(0), dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sc_ms, so_ms, ga_ms = (float(x) for x in tt.cpu())
        if rank == 0:
            sent = int(b.qp.nbytes) * (world - 1)
            recvd = int(d_sol.numel() * 8) * (world - 1)
            same = bool(torch.equal(allsol[:nb], allsol[nb:2 * nb]))       # every rank solved a copy of rank 0's batch
            sg = {"value": nb * world / ((sc_ms + so_ms + ga_ms) * 1e-3), "unit": UNIT, "scatter_ms": sc_ms, "solve_ms": so_ms, "gather_ms": ga_ms,
                  "bytes_scattered": sent, "bytes_gathered": recvd, "scatter_gbs_out_of_rank0": sent / (sc_ms * 1e-3) / 1e9,
                  "gather_gbs_into_rank0": recvd / (ga_ms * 1e-3) / 1e9, "backend": "nccl send/recv (acados_b200/sharding.py)",
                  "shards_identical_across_ranks": same}
        del full

    # ---- the north_star's target point: 65 536 QPs on 8 GPUs = 8192 per GPU (device-resident, same timing rules); run when the
    # job has 8 ranks, or on request (--target-batch).  The records are the rank's batch twice (the solve does not care).
    target = None
    tb = args.target_batch or (8192 if world == 8 else 0)
    if tb and tb % nb == 0 and tb > nb:
        solver3 = CuipmSolver(b.shape, tb, device=local_rank)
        solver3.set_tuning("fast", args.fast)
        d_qp3 = d_qp.repeat(tb // nb, 1)
        d_sol3 = torch.zeros((tb, b.layout.sol_stride), dtype=torch.float64, device="cuda")
        d_info3 = torch.zeros(tb * INFO_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
        st3 = torch.cuda.ExternalStream(solver3.lib.cuipm_stream(solver3.handle), device=torch.device("cuda", local_rank))
        for _ in range(2):
            solver3.solve_device(tb, d_qp3.data_ptr(), d_sol3.data_ptr(), d_info3.data_ptr(), opts, sync=False)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(st3):
            e0.record()
        nst = max(2, min(steps, 5))
        for _ in range(nst):
            solver3.solve_device(tb, d_qp3.data_ptr(), d_sol3.data_ptr(), d_info3.data_ptr(), opts, sync=False)
        with torch.cuda.stream(st3):
            e1.record()
        barrier()
        t3 = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        i3 = np.frombuffer(d_info3.cpu().numpy().tobytes(), dtype=INFO_DTYPE)
        target = {"global_batch": tb * world, "batch_per_gpu": tb, "value": tb * world * nst / (float(t3.item()) * 1e-3), "unit": UNIT,
                  "steps": nst, "ms_per_step": float(t3.item()) / nst, "all_converged": bool((i3["status"] == 0).all()),
                  "records": f"the rank's {nb} QPs {tb // nb} times"}
        solver3.close()
        del d_qp3, d_sol3, d_info3

    t = torch.tensor([dev_ms, e2e_s * 1e3, kernel_ms, solve_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, kernel_ms, solve_ms = (float(x) for x in t.cpu())
    total_qps = nb * world * steps
    value = total_qps / (dev_ms * 1e-3)
    e2e_value = total_qps / (e2e_ms * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        fp64 = {}
        try:
            fp64 = json.load(open(os.path.join(ROOT, "profiles", "r02_fp64_peak.json")))
        except Exception:
            pass
        fp64_peak = float(fp64.get("dfma_tflops", 33.9))
        ab = algorithmic_bytes_per_qp(b)
        achieved = ab["B_min"] * nb / (kernel_ms * 1e-3) / 1e9
        stream_gbs = ab["B_stream_iter"] * iters_mean * nb / (kernel_ms * 1e-3) / 1e9
        tflops = flops_per_qp(b, iters_mean) * nb / (kernel_ms * 1e-3) / 1e12
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        ncu = {}
        tp = os.path.join(ROOT, "profiles", "r02_ncu_headline.json")
        if os.path.exists(tp):
            try:
                ncu = json.load(open(tp))
            except Exception:
                ncu = {}
        if traffic is None:
            traffic = ncu.get("dram_bytes_per_launch")
        if _CONFIG != "c2" or nb != 4096:       # the committed ncu capture is of the headline configuration
            traffic, ncu = None, {}
        # SURVEY 8(d): the path is bounded by the FP64 pipe or by HBM; frac = the larger of the two fractions.  HBM term on
        # ALGORITHMIC bytes (B_min: every record read once, the solution written once), FP64 term on algorithmic flops against
        # the DFMA rate measured on this GPU type (scripts/ubench_fp64.cu -> profiles/r02_ubench_fp64.txt).
        frac_hbm, frac_fp64 = achieved / hbm_peak, tflops / fp64_peak
        roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": max(frac_hbm, frac_fp64),
                    "frac_hbm_algorithmic": frac_hbm, "frac_fp64_algorithmic": frac_fp64, "frac_is": "fp64" if frac_fp64 > frac_hbm else "hbm",
                    "traffic": traffic, "kernel": ("cuipm_fast_kernel (ring loop + first launch of the iteration-sliced scheduling)" if launches_per_step > 3 else "cuipm_fast_kernel") if args.fast and launches_per_step > 1 else "cuipm_solve_kernel",
                    "kernel_ms": kernel_ms, "solve_ms_all_kernels": solve_ms,
                    "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (of fallback)",
                    "algorithmic_bytes_per_qp": ab["B_min"], "mean_ipm_iterations": iters_mean,
                    "stream_model": {"bytes_per_qp": ab["B_stream_iter"] * iters_mean, "achieved_gbs": stream_gbs, "frac": stream_gbs / hbm_peak},
                    "fp64": {"achieved_tflops": tflops, "peak_tflops": fp64_peak,
                             "peak_source": "measured DFMA rate, profiles/r02_ubench_fp64.txt" if fp64 else "33.9 TFLOP/s (measured earlier on a B200 of this pool)",
                             "frac": frac_fp64, "ncu_pipe_fp64_cycles_active_pct": ncu.get("sm__pipe_fp64_cycles_active_pct")},
                    "ncu": ncu or None}
        cpu, parity = None, None
        if not args.no_cpu:
            try:
                nsamp = args.cpu_sample or nb
                cpu, rsol, rinfo = cpu_reference(b, opts, nsamp)
                # parity of the CUDA solutions of the same instances against the reference (untimed)
                gsol = h_sol.numpy()[:nsamp]
                du = np.max(np.abs(b.layout.u_traj(gsol) - b.layout.u_traj(rsol)), axis=1)
                parity = {"against": cpu["kind"], "instances": int(nsamp), "max_abs_du": float(du.max()),
                          "frac_du_le_1e-10": float((du <= 1e-10).mean()),
                          "iter_equal_frac": float((hinfo["iter"][:nsamp] == rinfo["iter"]).mean()),
                          "status_equal_frac": float((hinfo["status"][:nsamp] == rinfo["status"]).mean()),
                          "iter_mean_reference": float(rinfo["iter"].mean())}
                parity["iter_hist_cuda"] = np.bincount(hinfo["iter"][:nsamp]).tolist()
                parity["iter_hist_reference"] = np.bincount(rinfo["iter"]).tolist()
                if not args.no_tight:
                    # BASELINE.md section 4: second pass with all tolerances 1e-12 on the same instances, for the 1e-10 comparison
                    # (at the default tolerances both solvers stop ~1e-8 from the solution and round-off decides the last digits)
                    from oracle import oracle_binding as ob
                    from acados_b200.problems import Batch
                    topts = default_opts(res_g_max=1e-12, res_b_max=1e-12, res_d_max=1e-12, res_m_max=1e-12)
                    tsol, tinfo = solver.solve(b.qp[:nsamp], topts)
                    sub = Batch(b.shape, b.layout, np.ascontiguousarray(b.qp[:nsamp]), b.name)
                    if ob.have_ref():
                        trsol, trinfo, _ = ob.ref_solve(sub, topts, nthreads=host_threads())
                    else:
                        trsol, trinfo = ob.oracle_solve(sub, topts, nthreads=host_threads())
                    tdu = np.max(np.abs(b.layout.u_traj(tsol) - b.layout.u_traj(trsol)), axis=1)
                    parity["tight_1e-12"] = {"instances": int(nsamp), "max_abs_du": float(tdu.max()), "frac_du_le_1e-10": float((tdu <= 1e-10).mean()),
                                             "iter_equal_frac": float((tinfo["iter"] == trinfo["iter"]).mean()),
                                             "iter_within_one_frac": float((np.abs(tinfo["iter"] - trinfo["iter"]) <= 1).mean()),
                                             "status_hist_cuda": np.bincount(tinfo["status"], minlength=5).tolist(),
                                             "status_hist_reference": np.bincount(trinfo["status"], minlength=5).tolist(),
                                             "iter_hist_cuda": np.bincount(tinfo["iter"]).tolist(),
                                             "iter_hist_reference": np.bincount(trinfo["iter"]).tolist()}
            except Exception as e:  # noqa: BLE001
                cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": str(e)}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": dev_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(b.qp.nbytes) * world,
                        "d2h_bytes_per_step": int(h_sol.numel() * 8 + h_info.numel()) * world, "ms_per_step": e2e_ms / steps,
                        "lanes": 2, "chunks_per_call": args.e2e_pipe or 8,
                        "note": "two solver objects alternate (cuipm_solve_host_async / cuipm_wait): the copies of step i+1 overlap the solve "
                        "of step i; every call moves its whole batch in one piece (tuning key pipe=1) so that the solve runs with the "
                        "iteration-sliced scheduling (8 chunks per call -- the default, best for a single blocking call -- give 88 k QP/s here)"},
                "e2e_plugin": plugin, "scatter_gather": sg, "target_point": target,
                "gpu_launches": steps * launches_per_step,
                "roofline": roofline, "cpu_baseline": cpu, "parity": parity,
                "solver": {"status_hist": np.bincount(hinfo["status"], minlength=5).tolist(), "iter_mean": iters_mean,
                           "iter_max": int(info["iter"].max()), "lq_count": int(info["lq_count"].sum()),
                           "throughput_kernel": bool(args.fast and launches_per_step > 1), "launches_per_step": launches_per_step,
                           "handed_back_to_generic_kernel": handed_back}}
        real_stdout.write(json.dumps(line) + "\n"); real_stdout.flush()
    solver.close()
    solver2.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
