"""Batched get_best_theta_to_current_joints (r2ik_symik_best_theta_f64) against its cost model, the K = 33 sweep.

The search evaluates get_joints 33 times per searching pose (the preferred angle, then 16 iterations of two), so a
33-angle sweep of the same poses (r2ik_symik_sweep_f64, sampled angles, joints + state only) does the same number of
get_joints per pose with one solve each, and is the yardstick the search should approach.  For each arm, N poses
FK-sampled with current joints = the sampling joints + N(0, 0.3) noise, each solve kind, in one process:
  best_theta  r2ik_symik_best_theta_f64 (state + theta + joints)
  sweep33     r2ik_symik_sweep_f64, K = 33, on the same poses
  oracle      the CPU oracle's search (tests/hostsim/best_theta_oracle.c) on all host threads
Kernel times are CUDA-event medians of `--rounds` windows of `--reps` launches after warm-up; the oracle is timed once.

    python scripts/experiments/exp_best_theta.py [--lib path/to/libr2ik.so] [--out profiles/....json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
sys.path.insert(0, os.path.join(REPO, "tests"))

SIZES = [1024, 65536, 1 << 20]
K_SWEEP = 33


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None, help="another build of libr2ik.so (default: the in-tree library)")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--no-oracle", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from reachy2_symbolic_ik_b200 import _native, build

    if a.lib:
        _native.use_library(a.lib)
    else:
        build.build()
    import torch

    import best_theta_util as B
    from oracle import oracle
    from reachy2_symbolic_ik_b200 import SymbolicIK, _abi, fk

    orc = None
    if not a.no_oracle:
        _, orc = B.build_libs(tempfile.mkdtemp(prefix="exp_best_theta_"))
        threads = oracle.use_all_host_threads()
    header = {"card_name_power_limit": card(), "lib": a.lib or "in-tree", "reps": a.reps, "rounds": a.rounds,
              "oracle_threads": None if a.no_oracle else threads}
    print(json.dumps(header), flush=True)
    p = lambda t: C.c_void_p(None if t is None else t.data_ptr())   # noqa: E731
    i64, i32 = C.c_int64, C.c_int32
    MAT4 = _abi.POSE_MAT4
    rows = []
    for arm in B.ARMS:
        sv = SymbolicIK(arm=arm)
        lib, h, dev = sv._handle.lib, sv._handle.h, sv._device
        s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        pref = B.preferred_theta(arm)

        def timed(fn):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            ts = []
            for _ in range(a.rounds):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / a.reps)
            return float(np.median(ts)), float(min(ts)), float(max(ts))

        for n in SIZES:
            rng = np.random.default_rng(n + (arm == "l_arm"))
            q = fk.sample_fk_joints(n, rng)
            cj_np = q + rng.normal(scale=0.3, size=q.shape)
            P = fk.forward_kinematics_device(torch.as_tensor(q, device=dev), arm).reshape(n, 16).contiguous()
            cj = torch.as_tensor(cj_np, device=dev).contiguous()
            state = torch.empty(n, dtype=torch.uint8, device=dev)
            theta = torch.empty(n, dtype=torch.float64, device=dev)
            joints = torch.empty((n, 7), dtype=torch.float64, device=dev)
            sw_state = torch.empty(n, dtype=torch.uint8, device=dev)
            sw_j = torch.empty((n, K_SWEEP, 7), dtype=torch.float64, device=dev)
            for no_limits in (0, 1):
                def run_bt():
                    return lib.r2ik_symik_best_theta_f64(h, MAT4, p(P), i64(n), p(cj), i32(7), C.c_double(pref),
                                                         i32(no_limits), p(state), p(theta), p(joints), s)

                def run_sweep():
                    return lib.r2ik_symik_sweep_f64(h, MAT4, p(P), i64(n), None, i32(0), i32(K_SWEEP), i32(no_limits), None,
                                                    p(sw_state), None, None, p(sw_j), None, None, s)

                assert run_bt() == 0 and run_sweep() == 0, lib.r2ik_last_error()
                torch.cuda.synchronize()
                t_bt = timed(run_bt)
                t_sw = timed(run_sweep)
                ok = (state == 0)
                searched = ok & (theta != pref)
                r = {"arm": arm, "N": n, "no_limits": no_limits, "best_theta_ms": t_bt[0], "best_theta_min_max": t_bt[1:],
                     "sweep33_ms": t_sw[0], "sweep33_min_max": t_sw[1:], "best_theta_over_sweep33": t_bt[0] / t_sw[0],
                     "reachable": float(ok.float().mean().item()), "searched": float(searched.float().mean().item())}
                if orc is not None:
                    Pn = P.cpu().numpy()
                    t0 = time.perf_counter()
                    want = B.oracle_best_theta(orc, oracle, arm, Pn, cj_np, pref=pref, no_limits=bool(no_limits))
                    r["oracle_s"] = time.perf_counter() - t0
                    th = theta.cpu().numpy()
                    w = want[1]
                    r["theta_equal_oracle"] = float(np.mean((th == w) | (np.isnan(th) & np.isnan(w))))
                rows.append(r)
                print(json.dumps(r), flush=True)
            del P, cj, state, theta, joints, sw_state, sw_j
            torch.cuda.empty_cache()
    print(f"\n{header['card_name_power_limit']}  lib={header['lib']}  oracle threads={header['oracle_threads']}")
    print(f"{'arm':>5} {'N':>8} {'nl':>2} {'best ms':>9} {'sweep33':>9} {'ratio':>6} {'reach':>6} {'search':>6} "
          f"{'oracle s':>9} {'=oracle':>8}")
    for r in rows:
        print(f"{r['arm']:>5} {r['N']:>8} {r['no_limits']:>2} {r['best_theta_ms']:>9.4f} {r['sweep33_ms']:>9.4f} "
              f"{r['best_theta_over_sweep33']:>6.2f} {r['reachable']:>6.3f} {r['searched']:>6.3f} "
              f"{r.get('oracle_s', float('nan')):>9.3f} {r.get('theta_equal_oracle', float('nan')):>8.5f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"header": header, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
