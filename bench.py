#!/usr/bin/env python
"""bench.py -- benchmarks of the Reachy2 symbolic IK hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|symik|symik_f32|discrete|continuous|reachmap]
                    [--dump-outputs DIR]

The headline workload `symik` = BASELINE.json configs[1], the configuration the metric is quoted on: 1 M FK-sampled poses per
arm (r_arm and l_arm), FP64, reachability flag + theta interval + 7 joints at theta_interval[0] + elbow position.  One *step* =
one pass of K1 (`r2ik_symik_solve_f64`) over both arms' batches = 2 M solves per GPU; exactly K steps are timed.  With the
default `--workload all` the same JSON line also carries `workloads`: one sub-record per other BASELINE config -- `symik_f32`
(configs[1] on the FP32 fast path), `discrete` (configs[2], K = 360), `continuous` (configs[3], 65 536 x 1 000) and `reachmap`
(configs[4], 256^3 x 512, orientation-sharded over the ranks with the all-reduce timed separately) -- each with its own value,
ms_per_step, roofline, parity and e2e, under torchrun too, so that the scaling run measures every config at every N.

* own arm: `value` = poses/s with inputs resident in HBM (CUDA events on the launching stream, max over ranks); `e2e` = the
  same metric through the public facade with pinned HOST buffers, H2D and D2H copies inside the timed region (`e2e.lean`: the
  reference's own (N,6) input format and the state + joints record, 105 instead of 226 bytes per pose over the link);
  `roofline` for the dominant kernel; `cpu_baseline` = the C oracle (a port of the reference algorithm, OpenMP on all host
  threads) and, when `baseline/_ref` holds the installed Python reference, the reference itself on a bounded sample with one
  process per core; `scalar_latency` = what one control tick costs through the reference's scalar API.
* `--impl reference`: the reference algorithm's CPU implementation (oracle port, all host threads) on the same workloads;
  rank 0 only.
* N > 1: launched by torchrun, one rank per GPU, contiguous slices of the batch per rank, no data-path collective (weak
  scaling); the reach map shards orientations and all-reduces the count volume (strong scaling).
* `--dump-outputs DIR`: after the timed steps, rank 0 writes what the headline workload's last timed step gave it (under
  torchrun its slice of the batch; the all-reduced volume for the reach map) to
  DIR/<name>.npy, finite values only (NaN / inf entries as 0, marked in DIR/<name>_nonfinite.npy), a fixed sample of rows
  when the outputs exceed 48 MiB.  The inputs are seeded, so two builds run with the same arguments can be compared output
  for output.

The benchmark writes nothing into the source tree (it may be read-only): no bytecode cache, no build.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

sys.dont_write_bytecode = True   # the package, the oracle and the scripts it imports live in the (possibly read-only) tree
REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "ik_poses_per_sec"
UNIT = "poses/s"
ARMS = ("r_arm", "l_arm")


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for k, nme in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# =================================================================================================
# Python reference (baseline/_ref, pip-installed unmodified) on a bounded sample, one process per core
# =================================================================================================
def _pyref_available():
    return os.path.isdir(os.path.join(REPO, "baseline", "_ref", "reachy2_symbolic_ik"))


def _pyref_worker(args):
    kind, arm, poses = args
    import contextlib
    import io
    import warnings

    sys.path.insert(0, os.path.join(REPO, "baseline", "_ref"))
    warnings.filterwarnings("ignore")
    with contextlib.redirect_stdout(io.StringIO()):
        from reachy2_symbolic_ik.control_ik import ControlIK
        from reachy2_symbolic_ik.symbolic_ik import SymbolicIK
        from reachy2_symbolic_ik.utils import get_euler_from_homogeneous_matrix

        from reachy2_symbolic_ik_b200 import fk

        t0 = time.perf_counter()
        if kind == "symik":
            ik = SymbolicIK(arm=arm)
            for M in poses:
                goal = np.array(get_euler_from_homogeneous_matrix(M))  # (position, euler xyz), the reference's goal_pose
                ok, itv, f, _ = ik.is_reachable(goal)
                if ok:
                    f(itv[0])
        elif kind == "discrete":
            ctl = ControlIK(urdf=open(fk.bundled_urdf_path()).read())
            ctl.nb_search_points = 360
            for M in poses:
                ctl.symbolic_inverse_kinematics(arm, M, "discrete")
        elif kind == "continuous":
            for traj in poses:
                ctl = ControlIK(urdf=open(fk.bundled_urdf_path()).read())
                for M in traj:
                    ctl.symbolic_inverse_kinematics(arm, M, "continuous")
        return time.perf_counter() - t0


def python_reference_baseline(kind: str, arm: str, poses: np.ndarray, units: int):
    """poses: per-process work items are contiguous chunks.  Returns the `python_reference` sub-object."""
    if not _pyref_available():
        return None
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    chunks = [c for c in np.array_split(poses, cores) if len(c)]
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(len(chunks)) as pool:
        busy = pool.map(_pyref_worker, [(kind, arm, c) for c in chunks])
    wall = time.perf_counter() - t0
    return {"value": units / max(busy), "unit": UNIT, "cores": len(chunks), "kind": "reference",
            "per_core": units / sum(busy), "wall_s_incl_spawn": wall,
            "sample": f"unmodified pollen-robotics/reachy2_symbolic_ik (baseline/_ref) {kind}, {units} {arm} poses split over "
                      f"{len(chunks)} processes, numpy {np.__version__}"}


# =================================================================================================
# Workloads.  Each returns a dict of closures; all device work goes through the package facade / C ABI.
# =================================================================================================
class Symik:
    """configs[1]"""
    name = "symik"
    POSES_PER_ARM = 1_000_000
    SEEDS = {"r_arm": 1, "l_arm": 2}
    BYTES_IN, BYTES_OUT = 128, 1 + 1 + 16 + 56 + 24
    # FP64 flops the kernel executes per pose (FMA = 2): 272 DFMA + 176 DMUL + 125 DADD + 30 DSETP per pose, averaged over
    # the batch, in the ncu source-level counts of profiles/r1_s16 (DESIGN.md section 4).  SURVEY.md 8(d)'s weighted estimate
    # for the reference's formulation (library-cost transcendentals) is 2100 flop-equivalents; it is reported beside it.
    FLOP_EQ = 874.0
    FP64_PIPE_INSTR = 604.0   # DFMA + DMUL + DADD + DSETP per pose (profiles/r1_s43_symik_ncu_full.txt): pipe slots
    kernel = "k_symik_solve<MAT4>"
    e2e_extra_legs = ("lean", "goal_pose_input")

    def config(self, world):
        n = self.POSES_PER_ARM
        return {"workload": "configs[1]: 1M FK-sampled poses per arm (r_arm + l_arm), FP64, flag + theta interval + joints at "
                            "theta_interval[0] + elbow, (N,4,4) pose input", "poses_per_step_per_gpu": 2 * n,
                "global_poses_per_step": 2 * n * world, "pose_layout": "mat4_rowmajor_f64",
                "l2_policy": "inputs+outputs per step (452 MB) exceed the 126 MB L2; the two arms' batches alternate",
                "parallelism": f"pose-slices x{world}, no collective"}

    def host_poses(self, rank):
        from reachy2_symbolic_ik_b200 import fk

        return {arm: fk.sample_fk_poses(self.POSES_PER_ARM, arm, seed=self.SEEDS[arm] + 1000 * rank) for arm in ARMS}

    def setup(self, torch, dev, rank, world):
        from reachy2_symbolic_ik_b200 import SymbolicIK, _abi

        n = self.POSES_PER_ARM
        self.poses = self.host_poses(rank)
        self.solvers = {arm: SymbolicIK(arm=arm, device=dev.index) for arm in ARMS}
        self.dpose = {arm: torch.from_numpy(self.poses[arm]).reshape(n, 16).to(dev) for arm in ARMS}
        self.outs = {arm: dict(reach=torch.empty(n, dtype=torch.uint8, device=dev), state=torch.empty(n, dtype=torch.uint8, device=dev),
                               interval=torch.empty((n, 2), dtype=torch.float64, device=dev),
                               joints=torch.empty((n, 7), dtype=torch.float64, device=dev),
                               elbow=torch.empty((n, 3), dtype=torch.float64, device=dev)) for arm in ARMS}
        self.kind = _abi.POSE_MAT4
        self.units_per_step = 2 * n
        self.units_per_launch = n

    def step(self):
        for arm in ARMS:
            o = self.outs[arm]
            self.solvers[arm].solve_into(self.dpose[arm], self.kind, None, None, o["reach"], o["state"], o["interval"], o["joints"], o["elbow"])
        return 2

    def outputs(self):
        names = {"reach": "reachable", "state": "state", "interval": "theta_interval", "joints": "joints", "elbow": "elbow"}
        return {f"{arm}_{names[k]}": t for arm in ARMS for k, t in self.outs[arm].items()}

    def e2e_setup(self, torch):
        n = self.POSES_PER_ARM
        self.host_in = {arm: torch.from_numpy(self.poses[arm]).reshape(n, 16).pin_memory() for arm in ARMS}
        self.host_out = {arm: self.solvers[arm].alloc_host_outputs(n) for arm in ARMS}
        return {"h2d_bytes_per_step": 2 * n * self.BYTES_IN, "d2h_bytes_per_step": 2 * n * self.BYTES_OUT,
                "path": "SymbolicIK.is_reachable_batch_host: pinned host -> chunked H2D / K1 / D2H on 3 streams"}

    def e2e_step(self, torch):
        # a step = both arms' batches: both are enqueued, then both are waited for (results in host memory at step end)
        for arm in ARMS:
            self.solvers[arm].is_reachable_batch_host(self.host_in[arm], self.host_out[arm], wait=False)
        for arm in ARMS:
            self.solvers[arm].wait_host()

    def e2e_check(self, torch):
        assert torch.equal(self.host_out["r_arm"].joints[:1000].nan_to_num(), self.outs["r_arm"]["joints"][:1000].cpu().nan_to_num())

    def _goal_poses_pinned(self, torch):
        """The workload in the reference's OWN input format: goal_pose = (position, xyz euler), 48 B / pose."""
        from scipy.spatial.transform import Rotation as R

        if not hasattr(self, "_gp_pinned"):
            self._gp_pinned = {}
            for arm in ARMS:
                M = self.poses[arm]
                gp = np.concatenate([M[:, :3, 3], R.from_matrix(M[:, :3, :3]).as_euler("xyz")], axis=1)
                self._gp_pinned[arm] = torch.from_numpy(np.ascontiguousarray(gp)).pin_memory()
        return self._gp_pinned

    def _e2e_leg(self, env, steps, host_in, host_out, bytes_in, bytes_out, path, **kw):
        torch = env.torch
        n = self.POSES_PER_ARM
        def step():
            for arm in ARMS:
                self.solvers[arm].is_reachable_batch_host(host_in[arm], host_out[arm], wait=False, **kw)
            for arm in ARMS:
                self.solvers[arm].wait_host()

        for _ in range(2):
            step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
        dt = env.max_over_ranks(time.perf_counter() - t0)
        got = host_out["r_arm"].joints[:100_000].numpy()
        ref = self.outs["r_arm"]["joints"][:100_000].cpu().numpy()
        both = np.isfinite(got).all(axis=1) & np.isfinite(ref).all(axis=1)
        dj = np.abs(got[both] - ref[both]).max(axis=1)
        return {"value": 2 * n * env.world * steps / dt, "unit": UNIT, "h2d_bytes_per_step": 2 * n * bytes_in,
                "d2h_bytes_per_step": 2 * n * bytes_out, "steps": steps, "path": path,
                "median_abs_joint_difference_vs_mat4_input_rad": float(np.median(dj)),
                "state_agreement_vs_mat4_input": float((host_out["r_arm"].state[:100_000].numpy() ==
                                                        self.outs["r_arm"]["state"][:100_000].cpu().numpy()).mean())}

    def e2e_goal_pose_input(self, env, steps):
        """The same solves fed in the reference's input format (48 B / pose instead of the 128 B of a 4x4 matrix); all five outputs."""
        return self._e2e_leg(env, steps, self._goal_poses_pinned(env.torch), self.host_out, 48, self.BYTES_OUT,
                             "SymbolicIK.is_reachable_batch_host on (N,6) goal poses (the reference's input format), all outputs")

    def e2e_lean(self, env, steps):
        """The lean host record: (N,6) goal poses in, state + joints out = 48 + 57 B / pose over the link."""
        ik = self.solvers["r_arm"]
        if not hasattr(self, "_lean_out"):
            self._lean_out = {arm: self.solvers[arm].alloc_host_outputs(self.POSES_PER_ARM, want=ik.LEAN) for arm in ARMS}
        return self._e2e_leg(env, steps, self._goal_poses_pinned(env.torch), self._lean_out, 48, 57,
                             "SymbolicIK.is_reachable_batch_host((N,6) goal poses, want=SymbolicIK.LEAN): state + joints back",
                             want=ik.LEAN)

    def teardown(self):
        for k in ("_gp_pinned", "_lean_out", "host_in", "host_out", "dpose", "outs"):
            self.__dict__.pop(k, None)

    def parity(self, torch):
        from oracle import oracle as O

        m = 100_000
        want = O.symik_batch(O.arm_config("r_arm"), self.poses["r_arm"][:m])
        o = self.outs["r_arm"]
        got_j, got_i, got_s = o["joints"][:m].cpu().numpy(), o["interval"][:m].cpu().numpy(), o["state"][:m].cpu().numpy()
        ej, ei = np.abs(got_j - want[3]), np.abs(got_i - want[1])
        return {"checked_poses": m, "state_mismatches": int((got_s != want[2]).sum()),
                "max_abs_err_joints_rad": float(np.nanmax(ej)), "p99.9_abs_err_joints_rad": float(np.nanquantile(ej, 0.999)),
                "max_abs_err_interval_rad": float(np.nanmax(ei)), "over_1e-9": int((np.nan_to_num(ej).max(axis=1) > 1e-9).sum()),
                "vs": "CPU oracle (pinned to the reference by tests/golden)"}

    def cpu_port(self, poses=None, repeats=3):
        from oracle import oracle as O

        if poses is None:
            if not hasattr(self, "_cpu_data"):
                self._cpu_data = self.host_poses(0)
            poses = self._cpu_data
        cfgs = {arm: O.arm_config(arm) for arm in ARMS}
        if not getattr(self, "_cpu_warm", False):
            O.symik_batch(cfgs["r_arm"], poses["r_arm"][:20000])  # warm-up (thread pool, page-in), once
            self._cpu_warm = True
        best = float("inf")
        for _ in range(repeats):
            t0 = time.perf_counter()
            for arm in ARMS:
                O.symik_batch(cfgs[arm], poses[arm])
            best = min(best, time.perf_counter() - t0)
        n = sum(len(poses[a]) for a in ARMS)
        what = "full per-GPU workload" if n == 2 * self.POSES_PER_ARM else "first poses of the per-GPU workload"
        return n / best, best, O.max_threads(), f"{what} ({n} poses: {n // 2} per arm), C oracle + OpenMP"

    def pyref(self):
        cores = os.cpu_count() or 1
        m = 400 * cores
        return python_reference_baseline("symik", "r_arm", self.poses["r_arm"][:m], m)


class SymikF32(Symik):
    """configs[1] on the FP32 fast path (north_star: optional, 1e-4 rad): float32 poses in, float32 results out."""
    name = "symik_f32"
    BYTES_IN, BYTES_OUT = 64, 1 + 1 + 8 + 28 + 12
    # executed flops per pose (FMA = 2) in the ncu source-level counts of profiles/r1_s16: 573 FP32 (145 FFMA + 134 FMUL +
    # 78 FADD + 71 FSETP) + 58 FP64 of the mixed-precision front end (11 DFMA + 10 DMUL + 20 DADD + 6 DSETP)
    FLOP_EQ = 58.0       # FP64 part (roofline_fp64)
    FLOP_FP32 = 573.0    # FP32 part (roofline_fp32)
    kernel = "k_zero_u32 + k_symik_solve_f32<MAT4> + k_symik_escalated_f32<MAT4>"
    KERNELS_PER_PASS = 3      # the roofline's "launch" is one arm's pass: count reset, FP32 solve, FP64 re-solve of the escalated poses
    fp32 = True
    FP64_PIPE_INSTR = None
    e2e_extra_legs = ()

    def config(self, world):
        c = super().config(world)
        c["workload"] = c["workload"].replace("FP64", "FP32 fast path (FP64 front end + FP64 re-solve of undecidable poses)")
        c["pose_layout"] = "mat4_rowmajor_f32"
        c["l2_policy"] = "inputs+outputs per step (228 MB) exceed the 126 MB L2; the two arms' batches alternate"
        return c

    def host_poses(self, rank):
        return {arm: v.astype(np.float32) for arm, v in super().host_poses(rank).items()}

    def setup(self, torch, dev, rank, world):
        from reachy2_symbolic_ik_b200 import SymbolicIK, _abi

        n = self.POSES_PER_ARM
        self.poses = self.host_poses(rank)
        self.solvers = {arm: SymbolicIK(arm=arm, device=dev.index) for arm in ARMS}
        self.dpose = {arm: torch.from_numpy(self.poses[arm]).reshape(n, 16).to(dev) for arm in ARMS}
        f32 = torch.float32
        self.outs = {arm: dict(reach=torch.empty(n, dtype=torch.uint8, device=dev), state=torch.empty(n, dtype=torch.uint8, device=dev),
                               interval=torch.empty((n, 2), dtype=f32, device=dev), joints=torch.empty((n, 7), dtype=f32, device=dev),
                               elbow=torch.empty((n, 3), dtype=f32, device=dev)) for arm in ARMS}
        self.n_esc = torch.zeros(1, dtype=torch.int32, device=dev)
        self.esc = torch.empty(n, dtype=torch.int32, device=dev)
        self.kind = _abi.POSE_MAT4
        self.units_per_step = 2 * n
        self.units_per_launch = n

    def step(self):
        for arm in ARMS:
            o = self.outs[arm]
            self.solvers[arm].solve_into_f32(self.dpose[arm], self.kind, None, None, o["reach"], o["state"], o["interval"], o["joints"],
                                             o["elbow"], self.n_esc, scratch=self.esc)
        return 2

    def e2e_setup(self, torch):
        n = self.POSES_PER_ARM
        self.host_in = {arm: torch.from_numpy(self.poses[arm]).reshape(n, 16).pin_memory() for arm in ARMS}
        self.host_out = {arm: self.solvers[arm].alloc_host_outputs(n, "fp32") for arm in ARMS}
        return {"h2d_bytes_per_step": 2 * n * self.BYTES_IN, "d2h_bytes_per_step": 2 * n * self.BYTES_OUT,
                "path": "SymbolicIK.is_reachable_batch_host(precision='fp32'): pinned host -> chunked H2D / K1-f32 / D2H on 3 streams"}

    def e2e_step(self, torch):
        for arm in ARMS:
            self.solvers[arm].is_reachable_batch_host(self.host_in[arm], self.host_out[arm], precision="fp32", wait=False)
        for arm in ARMS:
            self.solvers[arm].wait_host()

    def parity(self, torch):
        from oracle import oracle as O

        m = 100_000
        o = self.outs["r_arm"]
        self.solvers["r_arm"].solve_into_f32(self.dpose["r_arm"], self.kind, None, None, o["reach"], o["state"], o["interval"],
                                             o["joints"], o["elbow"], self.n_esc, scratch=self.esc)
        esc = int(self.n_esc.item())
        want = O.symik_batch(O.arm_config("r_arm"), self.poses["r_arm"][:m].astype(np.float64))
        got_j, got_i, got_s = (o[k][:m].cpu().numpy() for k in ("joints", "interval", "state"))
        ej, ei = np.nan_to_num(np.abs(got_j - want[3])).max(axis=1), np.nan_to_num(np.abs(got_i - want[1])).max(axis=1)
        ok = want[2] == 0
        return {"checked_poses": m, "state_mismatches": int((got_s != want[2]).sum()),
                "stated_bound": "1e-4 rad for >= 99.99 % of the poses, 3e-4 rad for all (include/r2ik.h)",
                "max_abs_err_joints_rad": float(ej.max()), "p50_abs_err_joints_rad": float(np.median(ej[ok])),
                "p99.9_abs_err_joints_rad": float(np.quantile(ej[ok], 0.999)), "p99.99_abs_err_joints_rad": float(np.quantile(ej[ok], 0.9999)),
                "max_abs_err_interval_rad": float(ei.max()),
                "over_1e-4": int((ej > 1e-4).sum()), "over_3e-4": int((ej > 3e-4).sum()), "escalated_to_fp64_fraction": esc / self.POSES_PER_ARM,
                "vs": "FP64 CPU oracle on the same float32 inputs widened to double"}

    def cpu_port(self, poses=None, repeats=3):
        if poses is not None:
            poses = {a: v.astype(np.float64) for a, v in poses.items()}
        return super().cpu_port(poses, repeats)

    def pyref(self):
        return None


class Discrete:
    """configs[2]"""
    name = "discrete"
    N = 1_000_000
    K = 360
    BYTES_IN, BYTES_OUT = 128, 56 + 3
    kernel = "k_disc_consts + k_disc_classify + k_disc_search + k_disc_finish"
    KERNELS_PER_PASS = 4      # the roofline's "launch" is the four-kernel pass of r2ik_ctl_discrete_compact_f64

    SEARCH_FRACTION = 0.80   # share of the FK-sampled poses whose preferred theta fails and that run the elbow search

    @property
    def FLOP_EQ(self):
        # solve + joints + safety chain ~2400 flops per pose; the analytic search evaluates 17 candidate samples (7 sincos of
        # 35 shared by the neighbours, two half-plane tests 8, theta_k 2, wrapped cost 10) plus 4 atan2 + 2 roots to locate them (~200): independent of K;
        # 80 % of the poses search (length of the search list, profiles/r2_experiments.md)
        return 2400.0 + self.SEARCH_FRACTION * (7 * 35.0 + 17 * 20.0 + 200.0)

    def config(self, world):
        return {"workload": f"configs[2]: ControlIK discrete, 1M FK-sampled r_arm poses x {self.K} elbow-theta samples, in-kernel "
                            "best-elbow selection + joints + safety checks", "poses_per_step_per_gpu": self.N,
                "global_poses_per_step": self.N * world, "nb_search_points": self.K,
                "l2_policy": "inputs+outputs per step (187 MB) exceed the 126 MB L2",
                "parallelism": f"pose-slices x{world}, no collective"}

    def setup(self, torch, dev, rank, world):
        from reachy2_symbolic_ik_b200 import ControlIK, fk

        self.poses = fk.sample_fk_poses(self.N, "r_arm", seed=3 + 1000 * rank)
        self.ctl = ControlIK(urdf_path="../config_files/reachy2.urdf", device=dev.index)
        self.ctl.nb_search_points = self.K
        self.dM = torch.from_numpy(self.poses).reshape(self.N, 16).to(dev)
        self.out = None
        self.units_per_step = self.N
        self.units_per_launch = self.N

    def step(self):
        self.out = self.ctl.symbolic_inverse_kinematics_batch("r_arm", self.dM, "discrete", out=self.out)
        return 1

    def outputs(self):
        return dict(zip(("joints", "reachable", "state", "emergency_bits"), self.out))

    def e2e_setup(self, torch):
        self.host_in = torch.from_numpy(self.poses).reshape(self.N, 16).pin_memory()
        self.e2e_out = self.ctl.alloc_host_outputs("discrete", self.N)
        return {"h2d_bytes_per_step": self.N * self.BYTES_IN, "d2h_bytes_per_step": self.N * (self.BYTES_OUT + 1),
                "path": "ControlIK.symbolic_inverse_kinematics_batch_host: pinned host -> chunked H2D / K2 / D2H on 3 streams"}

    def e2e_step(self, torch):
        self.ctl.symbolic_inverse_kinematics_batch_host("r_arm", self.host_in, "discrete", out=self.e2e_out)

    def e2e_check(self, torch):
        assert np.array_equal(np.asarray(self.e2e_out[0][:1000]), self.out[0][:1000].cpu().numpy())

    def _oracle(self, M):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk
        from reachy2_symbolic_ik_b200.urdf import get_ik_parameters_from_urdf

        params = get_ik_parameters_from_urdf(open(fk.bundled_urdf_path()).read(), ["r", "l"])
        cfg = O.arm_config("r_arm", ik_parameters=params, singularity_offset=-1.01)
        return O.ctl_discrete_batch(cfg, O.ControlParams(arm="r_arm", nb_search_points=self.K), M)

    def parity(self, torch):
        m = 50_000
        wj, wr, ws, we = self._oracle(self.poses[:m])
        j, r, s, e = (x[:m].cpu().numpy() for x in self.out)
        ej = np.abs(j - wj)
        return {"checked_poses": m, "state_mismatches": int((s != ws).sum()), "flag_mismatches": int((r != wr).sum()),
                "max_abs_err_joints_rad": float(ej.max()), "p99.9_abs_err_joints_rad": float(np.quantile(ej, 0.999)),
                "over_1e-9": int((ej.max(axis=1) > 1e-9).sum()), "vs": "CPU oracle (pinned to the reference by tests/golden)"}

    def cpu_port(self, poses=None, repeats=2):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk

        if poses is None:
            if not hasattr(self, "_cpu_data"):
                self._cpu_data = fk.sample_fk_poses(200_000, "r_arm", seed=3)
            poses = self._cpu_data
        M = poses[:200_000]
        self._oracle(M[:5000])
        best = float("inf")
        for _ in range(repeats):
            t0 = time.perf_counter()
            self._oracle(M)
            best = min(best, time.perf_counter() - t0)
        return len(M) / best, best, O.max_threads(), f"first {len(M)} poses of the workload, K={self.K}, C oracle + OpenMP"

    def pyref(self):
        cores = os.cpu_count() or 1
        m = 40 * cores
        return python_reference_baseline("discrete", "r_arm", self.poses[:m], m)


class Continuous:
    """configs[3]"""
    name = "continuous"
    T, W = 65_536, 1_000
    BYTES_IN, BYTES_OUT = 128, 56 + 2
    FLOP_EQ = 2550.0          # is_reachable 900 + 10-sample search 350 + get_joints 900 + safety 300 + continuity 100
    kernel = "k_cont_targets + k_cont_thetas + k_cont_raw_joints_codes + k_cont_finish_codes + k_cont_apply_windings"
    KERNELS_PER_PASS = 5      # the roofline's "launch" is the five-kernel pass (plus torch's 2 MB state reset copy, not counted)

    def config(self, world):
        return {"workload": f"configs[3]: ControlIK continuous, {self.T} trajectories x {self.W} waypoints (joint-space sinusoids "
                            "through FK), joint continuity + multi-turn unwrapping", "poses_per_step_per_gpu": self.T * self.W,
                "global_poses_per_step": self.T * self.W * world, "unit_note": "a pose = one waypoint",
                "l2_policy": "inputs+outputs per step (12.2 GB) exceed the 126 MB L2",
                "parallelism": f"trajectory-slices x{world}, no collective"}

    def setup(self, torch, dev, rank, world):
        from reachy2_symbolic_ik_b200 import ControlIK, fk

        self.ctl = ControlIK(urdf_path="../config_files/reachy2.urdf", device=dev.index)
        self.dM = fk.sinusoidal_trajectories_device(self.T, self.W, "r_arm", seed=4 + 1000 * rank, device=dev)
        from reachy2_symbolic_ik_b200 import _abi

        st0 = np.zeros(self.T, dtype=_abi.TRAJ_STATE_DTYPE)
        st0["init"] = 1                       # every step replays the trajectories from a fresh controller
        self.st0 = torch.from_numpy(st0.view(np.uint8).reshape(self.T, -1)).to(dev)
        self.st = self.st0.clone()
        self.out = None
        self.units_per_step = self.T * self.W
        self.units_per_launch = self.T * self.W

    def step(self):
        self.st.copy_(self.st0)
        self.out = self.ctl.symbolic_inverse_kinematics_batch("r_arm", self.dM, "continuous", states=self.st, out=self.out)
        return 1

    def outputs(self):
        import torch

        st = self.out[3]                                      # (T, 80) bytes of _abi.TRAJ_STATE_DTYPE per trajectory
        f64, i32 = st[:, :64].view(torch.float64), st[:, 64:].view(torch.int32)
        return {"joints": self.out[0], "reachable": self.out[1], "state": self.out[2], "final_previous_theta": f64[:, 0],
                "final_previous_sol": f64[:, 1:], "final_emergency_stop": i32[:, 2], "final_emergency_bits": i32[:, 3]}

    def e2e_setup(self, torch):
        # a bounded slice of the trajectories goes host -> device -> host each e2e step
        self.e2e_T = 8192
        self.host_in = self.dM[: self.e2e_T].cpu().pin_memory()
        self.e2e_out = self.ctl.alloc_host_outputs("continuous", (self.e2e_T, self.W))
        return {"h2d_bytes_per_step": self.e2e_T * self.W * self.BYTES_IN, "d2h_bytes_per_step": self.e2e_T * self.W * self.BYTES_OUT,
                "path": f"ControlIK.symbolic_inverse_kinematics_batch_host on {self.e2e_T} of the trajectories per step: pinned host -> "
                        "chunked H2D / K3 / D2H on 3 streams", "units_per_step": self.e2e_T * self.W}

    def e2e_step(self, torch):
        self.ctl.symbolic_inverse_kinematics_batch_host("r_arm", self.host_in, "continuous", out=self.e2e_out)

    def e2e_check(self, torch):
        # the host pipeline cuts the waypoint axis: joints agree with the one-shot call to rounding (tests/test_gpu_control.py)
        assert np.allclose(np.asarray(self.e2e_out[0][:16]), self.out[0][:16].cpu().numpy(), rtol=0, atol=1e-12, equal_nan=True)

    def _oracle(self, M):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk
        from reachy2_symbolic_ik_b200.urdf import get_ik_parameters_from_urdf

        params = get_ik_parameters_from_urdf(open(fk.bundled_urdf_path()).read(), ["r", "l"])
        cfg = O.arm_config("r_arm", ik_parameters=params, singularity_offset=-1.01)
        return O.ctl_continuous_batch(cfg, O.ControlParams(arm="r_arm"), M)

    def parity(self, torch):
        m = 64
        M = self.dM[:m].cpu().numpy()
        wj, wr, ws, _ = self._oracle(M)
        j, r, s = (x[:m].cpu().numpy() for x in self.out[:3])
        ej = np.abs(j - wj)
        over = ej.max(axis=2) > 1e-9
        # a waypoint whose own oracle answer moves by > 1e-10 rad when the trajectory is perturbed by 3e-13 is
        # ill-conditioned (tests/parity.py): the reference does not determine it to 1e-9 either
        ill = np.zeros_like(over)
        rng = np.random.default_rng(1234)
        for _ in range(2):
            pj = self._oracle(M + rng.uniform(-3e-13, 3e-13, size=M.shape))[0]
            ill |= np.abs(pj - wj).max(axis=2) > 1e-10
        return {"checked_poses": m * self.W, "state_mismatches": int((s != ws).sum()), "flag_mismatches": int((r != wr).sum()),
                "max_abs_err_joints_rad": float(ej.max()), "over_1e-9": int(over.sum()),
                "over_1e-9_well_conditioned": int((over & ~ill).sum()), "ill_conditioned_waypoints": int(ill.sum()),
                "max_abs_err_joints_rad_well_conditioned": float(np.where(ill[..., None], 0.0, ej).max()),
                "vs": "CPU oracle (pinned to the reference by tests/golden)"}

    def cpu_port(self, poses=None, repeats=1):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk

        Tn = 2048
        if not hasattr(self, "_cpu_data"):
            self._cpu_data = fk.sinusoidal_trajectories(Tn, self.W, "r_arm", seed=4)[0]
        M = self._cpu_data
        t0 = time.perf_counter()
        self._oracle(M)
        dt = time.perf_counter() - t0
        return Tn * self.W / dt, dt, O.max_threads(), f"{Tn} trajectories x {self.W} waypoints, C oracle + OpenMP over trajectories"

    def pyref(self):
        cores = os.cpu_count() or 1
        M = self.dM[:cores, :100].cpu().numpy()
        return python_reference_baseline("continuous", "r_arm", M, cores * 100)


class ReachMap:
    """configs[4]"""
    name = "reachmap"
    N, N_ORI = 256, 512
    BYTES_IN, BYTES_OUT = 0, 4.0 / 512
    # per (voxel, orientation): ~25 % of the voxels pass the orientation-independent early-outs; a live pair costs the
    # FP64 front end of reach_flag_mixed (wrist, distance, radicand: ~17 flops) and its FP32 in-plane test (~35 flops);
    # 3e-4 of the live pairs are re-decided by the all-FP64 flag solve (~230 flops, negligible on average)
    FLOP_EQ = 0.25 * 17.0
    FLOP_FP32 = 0.25 * 35.0
    fp32 = True
    dtype = "f64+f32"   # FP64 front end and escalation, FP32 linking test; integer counts identical to the all-FP64 kernel
    kernel = "k_reach_map"

    def config(self, world):
        return {"workload": f"configs[4]: workspace reachability map, {self.N}^3 voxel grid x {self.N_ORI} orientations, per-voxel "
                            "reachable counts; sharded over the ranks, NCCL all-reduce of the per-voxel counts",
                "poses_per_step_per_gpu": self.N ** 3 * self.N_ORI // world, "global_poses_per_step": self.N ** 3 * self.N_ORI,
                "l2_policy": "no input traffic (poses generated from indices); 64 MiB count volume written per step",
                "parallelism": f"interleaved voxel rows x{world} + slab-pipelined NCCL all-reduce(sum) of the live x-range as 16-bit counts" if world > 1 else "single GPU, no collective"}

    scaling = "strong"

    def setup(self, torch, dev, rank, world):
        from reachy2_symbolic_ik_b200 import SymbolicIK, fk

        self._torch, self._events = torch, []
        self.ik = SymbolicIK(arm="r_arm", device=dev.index)
        self.ori = torch.from_numpy(fk.fibonacci_orientations(self.N_ORI)).to(dev)
        self.out = torch.empty((self.N,) * 3, dtype=torch.int32, device=dev)
        self.dist = None
        if world > 1:
            import torch.distributed as dist

            self.dist = dist
        self.world = world
        self.units_per_step = self.N ** 3 * self.N_ORI // world   # bench multiplies by world
        self.units_per_launch = self.N ** 3 * self.N_ORI // world

    def step(self):
        torch = self._torch
        if self.world > 1:
            t = {}
            self.ik.reach_map(n=self.N, orientations_euler=self.ori, dist=self.dist, out=self.out, timing=t)
            self._events.append(t)
            return len(t["k"])
        e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        e[0].record()
        self.ik.reach_map(n=self.N, orientations_euler=self.ori, out=self.out)
        e[1].record()
        self._events.append({"t0": e[0], "t1": e[1], "k": [(e[0], e[1])]})
        return 1

    def outputs(self):
        return {"counts": self.out}

    def phase_times(self, env, steps):
        """Kernel time (sum of the slab kernels) and what the all-reduce adds to the step beyond it, by events on the
        launching stream (max over ranks); plus, once, the plain form: one all-reduce of the full int32 volume after the kernel."""
        ev = self._events[-steps:]
        step_ms = env.max_over_ranks(float(np.mean([t["t0"].elapsed_time(t["t1"]) for t in ev])))
        k_ms = env.max_over_ranks(float(np.mean([sum(a.elapsed_time(b) for a, b in t["k"]) for t in ev])))
        out = {"kernel_ms": k_ms, "collective_ms": max(step_ms - k_ms, 0.0) if env.world > 1 else 0.0,
               "collective_share_of_step": max(step_ms - k_ms, 0.0) / step_ms if env.world > 1 else 0.0}
        if env.world > 1:
            torch = self._torch
            xb = ev[-1]["exchanged_bytes"]
            out["collective"] = {"op": "all_reduce(SUM), one per slab, asynchronous: overlaps the next slab's kernel", "slabs": 4,
                                 "sharding": "orientation slices (every rank counts its slice of the orientation set for every voxel)",
                                 "wire_dtype": "uint16 counts, two per int32 lane", "bytes": xb, "full_int32_volume_bytes": 4 * self.N ** 3,
                                 "backend": "NCCL (torch.distributed)", "collective_ms_is": "step time minus the slab kernels' time: "
                                 "the part of the exchange that the kernels do not hide, plus the 16->32-bit widening pass"}
            ms = []
            for _ in range(3):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record()
                self.ik.reach_map(n=self.N, orientations_euler=self.ori, dist=self.dist, out=self.out, plain_allreduce=True, mark=e[1].record)
                e[2].record(); torch.cuda.synchronize()
                ms.append((e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2])))
            oms = []
            for _ in range(3):
                t = {}
                self.ik.reach_map(n=self.N, orientations_euler=self.ori, dist=self.dist, out=self.out, timing=t, shard="voxels")
                torch.cuda.synchronize()
                oms.append((t["t0"].elapsed_time(t["t1"]), sum(a.elapsed_time(b) for a, b in t["k"])))
            out["voxel_row_sharded_form"] = {"step_ms": env.max_over_ranks(float(np.mean([a for a, _ in oms[1:]]))),
                                             "kernel_ms": env.max_over_ranks(float(np.mean([b for _, b in oms[1:]]))),
                                             "note": "each rank counts all orientations for every world-th voxel row, the all-reduce adds disjoint "
                                                     "pieces; same 16-bit, live-range, slab-pipelined exchange"}
            out["plain_form"] = {"kernel_ms": env.max_over_ranks(float(np.mean([a for a, _ in ms[1:]]))),
                                 "collective_ms": env.max_over_ranks(float(np.mean([b for _, b in ms[1:]]))),
                                 "bytes": 4 * self.N ** 3, "note": "one all-reduce of the full int32 volume after the kernel (the round-1 form)"}
        return out

    def e2e_setup(self, torch):
        self.host_out = torch.empty((self.N,) * 3, dtype=torch.int32).pin_memory()
        return {"h2d_bytes_per_step": self.N_ORI * 24, "d2h_bytes_per_step": self.N ** 3 * 4,
                "path": "SymbolicIK.reach_map + D2H of the count volume"}

    def e2e_step(self, torch):
        self.ik.reach_map(n=self.N, orientations_euler=self.ori.cpu().numpy(), dist=self.dist, out=self.out)
        self.host_out.copy_(self.out, non_blocking=True)

    def e2e_check(self, torch):
        torch.cuda.synchronize()
        assert int(self.host_out.sum()) == int(self.out.sum())

    def parity(self, torch):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk, workspace

        n, no = 40, 32
        ori = fk.fibonacci_orientations(no)
        origin, step, dims = workspace.reach_grid(self.ik.shoulder_position, self.ik.max_arm_length, n)
        got = self.ik.reach_map(n=n, orientations_euler=ori).cpu().numpy()
        want = O.reach_map(O.arm_config("r_arm"), origin, step, dims, ori)
        d = got.astype(np.int64) - want.astype(np.int64)
        return {"checked_poses": n ** 3 * no, "voxels_differing": int((d != 0).sum()), "max_abs_count_diff": int(np.abs(d).max()),
                "reachable_total": int(want.sum()), "full_map_reachable_total": int(self.out.sum().item()),
                "vs": "CPU oracle on a 40^3 x 32 sub-problem"}

    def cpu_port(self, poses=None, repeats=1):
        from oracle import oracle as O
        from reachy2_symbolic_ik_b200 import fk, workspace

        n, no = 64, 64
        ori = fk.fibonacci_orientations(no)
        origin, step, dims = workspace.reach_grid([0.0, -0.2, 0.0], 0.66, n)
        t0 = time.perf_counter()
        O.reach_map(O.arm_config("r_arm"), origin, step, dims, ori)
        dt = time.perf_counter() - t0
        return n ** 3 * no / dt, dt, O.max_threads(), f"{n}^3 x {no} sub-grid of the same cube, C oracle + OpenMP, extrapolated linearly"

    def pyref(self):
        return None


WORKLOADS = {w.name: w for w in (Symik, SymikF32, Discrete, Continuous, ReachMap)}


def reference_record(wl, steps, warmup):
    """One workload on the CPU arm: `warmup` + `steps` passes of the C port over the bounded sample cpu_port() defines."""
    vals, secs = [], []
    sample = cores = None
    for _ in range(warmup):
        wl.cpu_port(repeats=1)
    for _ in range(steps):
        v, dt, cores, sample = wl.cpu_port(repeats=1)
        vals.append(v); secs.append(dt)
    value = float(np.mean(vals))
    return {"value": value, "unit": UNIT, "steps": steps, "warmup": warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": f"per step: {sample}"}}


def run_reference(args, names):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as O

    O.use_all_host_threads()   # torchrun exports OMP_NUM_THREADS=1
    head = WORKLOADS[names[0]]()
    if isinstance(head, Symik):
        # the headline workload honours --steps / --warmup exactly: the per-step sample shrinks instead (a step is a
        # pass of the CPU port over the first poses of the workload, about 40 M solves for the whole run)
        steps = args.steps or 10
        warmup = args.warmup if args.warmup is not None else 1
        per_arm = int(min(head.POSES_PER_ARM, max(10_000, 20_000_000 // (steps + warmup))))
        full = head.host_poses(0)
        head._cpu_data = {arm: full[arm][:per_arm] for arm in ARMS}
    else:
        # one reference step is a fraction of a second to a few seconds of all host cores: bound the run
        steps = min(args.steps or 10, 20)
        warmup = min(args.warmup if args.warmup is not None else 1, 2)
    rec = reference_record(head, steps, warmup)
    cfg = head.config(args.gpus)
    cfg["reference_sample"] = rec["cpu_baseline"]["sample"] + " (the CPU arm times a bounded sample of the workload, not all of it)"
    line = {
        "impl": "reference", "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
        "scaling": getattr(head, "scaling", "weak"), "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg, "cpu_baseline": rec["cpu_baseline"],
        "e2e": {"value": rec["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference is pure Python (NumPy/SciPy, single-threaded, ~1e3 poses/s/core, reported as cpu_baseline.python_reference); this arm times the C port of "
                "its algorithm (oracle/, pinned to the reference's outputs by tests/golden) on all host threads -- a much "
                "stronger CPU baseline than the reference itself.",
    }
    # the unmodified Python reference itself (baseline/_ref), on a bounded sample, beside the port
    pr = None
    try:
        if isinstance(head, Symik):
            from reachy2_symbolic_ik_b200 import fk

            m = 400 * (os.cpu_count() or 1)
            pr = python_reference_baseline("symik", "r_arm", fk.sample_fk_poses(m, "r_arm", seed=head.SEEDS["r_arm"]), m)
    except Exception as e:  # the installed reference is optional
        pr = {"unavailable": repr(e)}
    if pr is not None:
        line["cpu_baseline"]["python_reference"] = pr
    subs = {}
    for name in names[1:]:
        try:
            wl = WORKLOADS[name]()
            r = reference_record(wl, 2, 1)
            r["config"] = {"workload": wl.config(args.gpus)["workload"]}
            subs[name] = r
        except Exception as e:
            subs[name] = {"error": repr(e)}
    if subs:
        line["workloads"] = subs
    emit(line)
    return 0


_REAL_STDOUT = None


def claim_stdout() -> None:
    """stdout carries exactly ONE line (the JSON result): everything else that writes to file descriptor 1 -- the facade's
    reference-style prints, NCCL's version banner when NCCL_DEBUG is set -- is sent to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def csrc_sha16() -> str:
    """Identity of the kernel sources the loaded library was built from (the committed ncu captures carry the same tag)."""
    import hashlib

    h = hashlib.sha256()
    d = os.path.join(REPO, "reachy2_symbolic_ik_b200", "csrc")
    for f in sorted(os.listdir(d)):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


class Env:
    """Process-level context shared by the workloads of one run."""

    def __init__(self, torch, dist, dev, rank, world, local_rank):
        self.torch, self.dist, self.dev, self.rank, self.world, self.local_rank = torch, dist, dev, rank, world, local_rank

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.dist is None:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())


DUMP_BYTES = 48 << 20     # --dump-outputs writes at most this much (float32 / float64 .npy payloads)
DUMP_SEED = 0


def dump_outputs(wl, dirname: str) -> dict:
    """Write what the last timed step computed as <dirname>/<name>.npy: float arrays in their own precision, flags, states
    and counts as float32 (exact).  Every file holds finite values only: the solver returns NaN joints / interval / elbow
    for a pose it cannot reach, so each float output is written with those entries set to 0 beside
    <name>_nonfinite.npy (float32, 1 where the caller receives NaN or inf), which together say exactly what was returned.
    When the outputs exceed DUMP_BYTES, every array keeps the same fixed, seeded sample of rows along its first axis
    (poses, trajectories or voxel planes), sorted; arrays of equal length share the sample."""
    import torch

    outs = wl.outputs()
    total = sum(t.numel() * ({torch.float64: 8 + 4, torch.float32: 4 + 4}.get(t.dtype, 4)) for t in outs.values())
    frac = min(1.0, DUMP_BYTES / total)
    os.makedirs(dirname, exist_ok=True)
    rows = {}
    for name, t in outs.items():
        n = t.shape[0]
        k = int(n * frac)
        if k < n:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
            t = t.index_select(0, torch.from_numpy(idx).to(t.device))
        a = t.cpu().numpy()
        if a.dtype in (np.float32, np.float64):
            bad = ~np.isfinite(a)
            np.save(os.path.join(dirname, name + "_nonfinite.npy"), bad.astype(np.float32))
            a = np.where(bad, a.dtype.type(0), a)
        np.save(os.path.join(dirname, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float32))
        rows[name] = [k, n]
    return {"dir": os.path.abspath(dirname), "rows_written_of_total": rows, "sample_seed": DUMP_SEED if frac < 1.0 else None}


def run_workload(env: Env, wl, steps: int, warmup: int, cpu_baseline: bool, dump_dir: str | None = None):
    """Time one workload: W warm-up steps, exactly K timed steps (barrier + synchronize on both sides, CUDA events on the
    launching stream, max over ranks), the end-to-end leg, the parity spot check, the rooflines.  Returns the record.
    dump_dir: rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    import contextlib

    torch, dev, rank, world = env.torch, env.dev, env.rank, env.world
    from reachy2_symbolic_ik_b200 import _native

    with contextlib.redirect_stdout(sys.stderr):   # the facade prints like the reference ("Using default parameters")
        wl.setup(torch, dev, rank, world)
    for _ in range(warmup):
        wl.step()
    env.barrier()
    launches = 0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(env.local_rank) as clocks:
        ev0.record()
        for _ in range(steps):
            launches += wl.step()
        ev1.record()
        env.barrier()
    ms_total = env.max_over_ranks(ev0.elapsed_time(ev1))
    units_per_step = wl.units_per_step * world
    value = units_per_step * steps / (ms_total * 1e-3)
    kernel_ms = ms_total / launches  # a step is nothing but launches of the dominant kernel(s): average launch duration
    rec = {"value": value, "unit": UNIT, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
           "scaling": getattr(wl, "scaling", "weak"),
           "dtype": getattr(wl, "dtype", "f32" if getattr(wl, "fp32", False) else "f64"), "config": wl.config(world),
           "gpu_launches": launches * getattr(wl, "KERNELS_PER_PASS", 1), "clocks": clocks.summary()}
    if dump_dir is not None and rank == 0:     # before phase_times: under torchrun it runs the reach map again
        rec["dump_outputs"] = dict(dump_outputs(wl, dump_dir), rank=rank, world_size=world,
                                   covers="this rank's share of the step" if world > 1 else "the whole step")
    if hasattr(wl, "phase_times"):
        rec.update(wl.phase_times(env, steps))

    # ---- end to end through the public facade with pinned host buffers (copies inside the timed region)
    e2e_info = wl.e2e_setup(torch)
    e2e_units = e2e_info.pop("units_per_step", wl.units_per_step) * world
    for _ in range(2):
        wl.e2e_step(torch)
    env.barrier()
    e2e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        wl.e2e_step(torch)
    torch.cuda.synchronize()
    e2e_s = env.max_over_ranks(time.perf_counter() - t0)
    wl.e2e_check(torch)
    rec["e2e"] = {"value": e2e_units * e2e_steps / e2e_s, "unit": UNIT, **e2e_info, "steps": e2e_steps}
    for name in getattr(wl, "e2e_extra_legs", ()):
        try:     # optional legs: can only add a key
            rec["e2e"][name] = getattr(wl, "e2e_" + name)(env, e2e_steps)
        except Exception as e:
            rec["e2e"][name] = {"unavailable": repr(e)}

    # ---- parity spot check against the oracle on this rank's data (not timed), CPU baselines
    if rank == 0:
        rec["parity"] = wl.parity(torch)
        if world == 1 and cpu_baseline:
            from oracle import oracle as O

            O.use_all_host_threads()
            v, dt, cores, sample = wl.cpu_port(getattr(wl, "poses", None))
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
            try:
                pr = wl.pyref()
            except Exception as e:  # the installed reference is optional
                pr = {"unavailable": repr(e)}
            if pr is not None:
                cpu["python_reference"] = pr
            rec["cpu_baseline"] = cpu

    # ---- rooflines for the dominant kernel
    hbm_peak, peak_src = measured_peaks()
    alg_bytes = (wl.BYTES_IN + wl.BYTES_OUT) * wl.units_per_launch
    achieved_gbs = alg_bytes / (kernel_ms * 1e-3) / 1e9
    pms, pfl = C.c_double(), C.c_double()
    _native.check(_native.load().r2ik_dfma_probe(env.local_rank, 400000, C.byref(pms), C.byref(pfl), None), "r2ik_dfma_probe")
    fp64_peak = pfl.value / (pms.value * 1e-3) / 1e12
    # dram__bytes_read + dram__bytes_write of one launch and the pipe activity, from the committed ncu --set full capture of
    # this kernel (scripts/ncu_to_json.py -> profiles/<workload>_ncu.json); null when no capture is committed
    traffic = ncu = None
    tp = os.path.join(REPO, "profiles", f"{wl.name}_ncu.json")
    if os.path.exists(tp):
        with open(tp) as f:
            ncu = json.load(f)
        traffic = ncu.get("dram_bytes_per_launch")
    hbm = {"bound": "hbm", "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
           "traffic": traffic, "kernel": wl.kernel, "kernel_ms": kernel_ms,
           "algorithmic_bytes_per_pose": wl.BYTES_IN + wl.BYTES_OUT, "poses_per_launch": wl.units_per_launch,
           "peak_source": peak_src,
           "traffic_source": None if ncu is None else {"file": f"profiles/{wl.name}_ncu.json", "capture": ncu.get("source"),
                                                       "csrc_sha16_of_capture": ncu.get("csrc_sha16"),
                                                       "csrc_sha16_running": csrc_sha16()}}
    # FP64 pipe: every FP64 instruction (DFMA, DADD, DMUL, DSETP) holds the pipe for the same two cycles per warp, so the
    # pipe roofline counts instructions (x 2 = DFMA-equivalent flops) against the measured DFMA peak.  Kernels without a
    # counted instruction mix fall back to their flop estimate (FMA = 2).
    slots = getattr(wl, "FP64_PIPE_INSTR", None)
    fp64_flop = 2.0 * slots if slots is not None else wl.FLOP_EQ
    fp64_ach = fp64_flop * wl.units_per_launch / (kernel_ms * 1e-3) / 1e12
    fp64 = {"bound": "fp64", "achieved": fp64_ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": fp64_ach / fp64_peak,
            "kernel": wl.kernel, "kernel_ms": kernel_ms,
            "accounting": ("FP64-pipe instructions per pose x 2 (DFMA-equivalent): the pipe issues one FP64 instruction of any kind "
                           "per two cycles per SM sub-partition" if slots is not None else "estimated FP64 flops per pose (FMA = 2)"),
            "fp64_pipe_instructions_per_pose": slots, "flop_per_pose": fp64_flop,
            "peak_source": "r2ik_dfma_probe measured in this run (DFMA chains, full grid)",
            "ncu": None if ncu is None else {k: ncu.get(k) for k in (
                "fp64_pipe_pct_of_peak", "issue_active_pct", "warps_active_pct", "registers_per_thread", "warp_instructions", "source")}}
    # Issue slots: every SM sub-partition issues at most one warp instruction per cycle.  The executed warp instructions of
    # one launch come from the committed ncu capture (a count, independent of the profiler's timing); the clock is the SM
    # clock sampled under load during the timed region (else the maximum clock).
    issue = None
    if ncu is not None and ncu.get("warp_instructions"):
        cl = rec["clocks"]
        mhz = cl.get("sm_mhz") or cl.get("sm_max_mhz")
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        if mhz:
            peak_ips = n_sm * 4 * mhz * 1e6
            ach_ips = ncu["warp_instructions"] / (kernel_ms * 1e-3)
            issue = {"bound": "issue", "achieved": ach_ips / 1e9, "peak": peak_ips / 1e9, "unit": "G warp-instructions/s",
                     "frac": ach_ips / peak_ips, "kernel": wl.kernel, "kernel_ms": kernel_ms,
                     "warp_instructions_per_launch": ncu["warp_instructions"], "sm_count": n_sm, "sm_mhz": mhz,
                     "accounting": "executed warp instructions of one launch (ncu smsp__inst_executed.sum of the committed capture) / measured "
                                   "launch time, against SMs x 4 sub-partitions x SM clock",
                     "ncu_issue_active_pct": ncu.get("issue_active_pct")}
    # `roofline` names the limiter that binds: the bound whose lower limit on the launch time is the largest
    cands = [hbm, fp64] + ([issue] if issue is not None else [])
    if getattr(wl, "fp32", False):
        cands.remove(fp64)          # mixed-precision kernels: the FP64 share is reported beside, it is not their limiter
    binding = max(cands, key=lambda r_: r_["frac"])
    rec["roofline"] = dict(binding)
    rec["roofline"]["traffic"] = traffic
    others = [r_ for r_ in (hbm, fp64, issue) if r_ is not None and r_ is not binding]
    rec["roofline"]["note"] = (f"every lower bound is reported; `roofline` is the binding one ({binding['bound']}: frac {binding['frac']:.3f}); "
                               "the others: " + ", ".join(f"roofline_{o['bound']} (frac {o['frac']:.3f})" for o in others))
    for o in others:
        rec["roofline_" + o["bound"]] = o
    if getattr(wl, "fp32", False):
        # mixed-precision kernels (K1-f32, K4): the measured FFMA peak beside the DFMA one
        _native.check(_native.load().r2ik_ffma_probe(env.local_rank, 400000, C.byref(pms), C.byref(pfl), None), "r2ik_ffma_probe")
        fp32_peak = pfl.value / (pms.value * 1e-3) / 1e12
        fp32_ach = wl.FLOP_FP32 * wl.units_per_launch / (kernel_ms * 1e-3) / 1e12
        rec["roofline_fp32"] = {"bound": "fp32", "achieved": fp32_ach, "peak": fp32_peak, "unit": "TFLOP/s",
                                "frac": fp32_ach / fp32_peak, "fp32_flop_per_pose": wl.FLOP_FP32,
                                "peak_source": "r2ik_ffma_probe measured in this run (FFMA chains, full grid)",
                                "note": "mixed-precision kernel: the FP32 flops are counted here, the FP64 flops in "
                                        "roofline_fp64; the two pipes issue from the same slots"}
    if hasattr(wl, "teardown"):
        wl.teardown()
    del wl
    torch.cuda.empty_cache()
    return rec


def scalar_latency():
    """One control tick through the reference's scalar API (examples call it once per tick, src/example/example_control.py:9-27)."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("exp_scalar", os.path.join(REPO, "scripts", "experiments", "exp_r2_scalar_latency.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod.measure(200)


SUB_STEPS = {"symik_f32": (50, 5), "discrete": (20, 5), "continuous": (3, 3), "reachmap": (3, 3)}   # (steps, warm-up) as sub-records


def main() -> int:
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline workload's last timed step to DIR/<name>.npy, NaN / inf as 0 and "
                         "marked in DIR/<name>_nonfinite.npy (about 48 MiB at most)")
    args = ap.parse_args()
    names = ["symik", "symik_f32", "discrete", "continuous", "reachmap"] if args.workload == "all" else [args.workload]
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU path's outputs; the reference arm keeps none")
        return run_reference(args, names)
    head = WORKLOADS[names[0]]()
    default_steps = {"symik": 2000, "symik_f32": 2000, "discrete": 50, "continuous": 5, "reachmap": 5}[head.name]
    default_warm = {"symik": 20, "symik_f32": 20, "discrete": 5, "continuous": 3, "reachmap": 3}[head.name]
    args.steps = args.steps or default_steps
    args.warmup = max(args.warmup if args.warmup is not None else default_warm, 3)

    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from reachy2_symbolic_ik_b200 import hostmem

    binding = hostmem.bind_to_gpu_numa(local_rank)     # pinned buffers and copy threads next to this rank's GPU
    env = Env(torch, dist, torch.device("cuda", local_rank), rank, world, local_rank)
    rec = run_workload(env, head, args.steps, args.warmup, cpu_baseline=not args.no_cpu_baseline, dump_dir=args.dump_outputs)
    subs = {}
    for name in names[1:]:
        k, w = SUB_STEPS[name]
        try:
            subs[name] = run_workload(env, WORKLOADS[name](), k, w, cpu_baseline=not args.no_cpu_baseline)
        except Exception as e:   # a sub-record can only add a key: the headline line stands without it
            import traceback

            traceback.print_exc()
            subs[name] = {"error": repr(e)}
        env.barrier()
    if rank == 0:
        line = {"metric": METRIC, "value": rec.pop("value"), "unit": rec.pop("unit"), "n_gpus": world, "steps": rec.pop("steps"),
                "warmup": rec.pop("warmup"), "ms_per_step": rec.pop("ms_per_step"), "higher_is_better": True,
                "scaling": rec.pop("scaling"), "vs_baseline": None, "dtype": rec.pop("dtype"), "data": "synthetic",
                "config": rec.pop("config"), **rec, "host_binding": binding}
        if subs:
            line["workloads"] = subs
            line["gpu_launches_all_workloads"] = line["gpu_launches"] + sum(v.get("gpu_launches", 0) for v in subs.values())
        if world == 1 and args.workload == "all":
            try:
                line["scalar_latency"] = scalar_latency()
            except Exception as e:
                line["scalar_latency"] = {"unavailable": repr(e)}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
