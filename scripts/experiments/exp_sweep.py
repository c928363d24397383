"""Elbow-angle sweep (r2ik_symik_sweep_f64) against the one-angle solve on the expanded batch.

For each shape (N poses x K angles), given and sampled angles, no_limits 0 and 1, in one process:
  sweep      r2ik_symik_sweep_f64 on N poses x K angles (joints + elbow + thetas_used + projected + state + interval)
  expanded   r2ik_symik_solve_f64 (no_limits: r2ik_symik_no_limits_f64) on the N*K-pose batch with the same angles
  model      K1 solve-only on N poses (joints = elbow = NULL) + K x (full K1 - solve-only K1) on N poses
and asserts that the sweep's joints / elbows (and states / intervals) equal the expanded batch's bit for bit.
Times are CUDA-event medians of `--rounds` windows of `--reps` launches after warm-up; every output array of the
sweep is larger than the 126 MB L2 at the default shapes.

    python scripts/experiments/exp_sweep.py [--lib path/to/libr2ik.so] [--out /tmp/exp_sweep.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)

SHAPES = [(1 << 20, 8), (65536, 128), (1024, 4096)]


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
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    from reachy2_symbolic_ik_b200 import _native, build

    if a.lib:
        _native.use_library(a.lib)
    else:
        build.build()
    import torch

    from reachy2_symbolic_ik_b200 import SymbolicIK, _abi, fk

    sv = SymbolicIK(arm="r_arm")
    lib, h, dev = sv._handle.lib, sv._handle.h, sv._device
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: C.c_void_p(None if t is None else t.data_ptr())   # noqa: E731
    i64, i32 = C.c_int64, C.c_int32
    MAT4 = _abi.POSE_MAT4

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

    def same(x, y):
        return bool(((x == y) | (torch.isnan(x) & torch.isnan(y))).all().item())

    rows = []
    header = {"card_name_power_limit": card(), "lib": a.lib or "in-tree", "reps": a.reps, "rounds": a.rounds}
    print(json.dumps(header), flush=True)
    gen = torch.Generator(device=dev).manual_seed(1234)
    for n, K in SHAPES:
        q = torch.as_tensor(fk.sample_fk_joints(n, np.random.default_rng(n)), device=dev)
        P = fk.forward_kinematics_device(q, "r_arm").reshape(n, 16).contiguous()
        del q
        state = torch.empty(n, dtype=torch.uint8, device=dev)
        itv = torch.empty((n, 2), dtype=torch.float64, device=dev)
        used = torch.empty((n, K), dtype=torch.float64, device=dev)
        j = torch.empty((n, K, 7), dtype=torch.float64, device=dev)
        el = torch.empty((n, K, 3), dtype=torch.float64, device=dev)
        proj = torch.empty((n, K), dtype=torch.uint8, device=dev)
        given = (torch.rand((n, K), generator=gen, device=dev, dtype=torch.float64) * 8 - 4).contiguous()
        # model terms: K1 on N poses, solve only and full (angle = the first column)
        k1_state = torch.empty(n, dtype=torch.uint8, device=dev)
        k1_itv = torch.empty((n, 2), dtype=torch.float64, device=dev)
        k1_j = torch.empty((n, 7), dtype=torch.float64, device=dev)
        k1_e = torch.empty((n, 3), dtype=torch.float64, device=dev)
        th0 = given[:, 0].contiguous()
        t_solve = timed(lambda: lib.r2ik_symik_solve_f64(h, MAT4, p(P), None, None, i64(n), None, p(k1_state), p(k1_itv),
                                                         None, None, s))
        t_full = timed(lambda: lib.r2ik_symik_solve_f64(h, MAT4, p(P), p(th0), None, i64(n), None, p(k1_state), p(k1_itv),
                                                        p(k1_j), p(k1_e), s))
        model = t_solve[0] + K * (t_full[0] - t_solve[0])
        Pe = P.repeat_interleave(K, dim=0).contiguous()
        ne = n * K
        e_state = torch.empty(ne, dtype=torch.uint8, device=dev)
        e_itv = torch.empty((ne, 2), dtype=torch.float64, device=dev)
        e_j = torch.empty((ne, 7), dtype=torch.float64, device=dev)
        e_e = torch.empty((ne, 3), dtype=torch.float64, device=dev)
        e_proj = torch.empty(ne, dtype=torch.uint8, device=dev)
        for no_limits in (0, 1):
            for mode in ("given", "sampled"):
                th = given if mode == "given" else None
                stride = K if th is not None else 0

                def run_sweep():
                    return lib.r2ik_symik_sweep_f64(h, MAT4, p(P), i64(n), p(th), i32(stride), i32(K), i32(no_limits), None,
                                                    p(state), p(itv), p(used), p(j), p(el), p(proj), s)

                assert run_sweep() == 0, lib.r2ik_last_error()
                torch.cuda.synchronize()
                angles = used.reshape(-1).contiguous()      # the angles the sweep used (NaN for an unreachable pose)
                if no_limits:
                    def run_exp():
                        return lib.r2ik_symik_no_limits_f64(h, MAT4, p(Pe), p(angles), None, i32(0), i64(ne), p(e_j), p(e_e),
                                                            p(e_proj), s)
                else:
                    def run_exp():
                        return lib.r2ik_symik_solve_f64(h, MAT4, p(Pe), p(angles), None, i64(ne), None, p(e_state), p(e_itv),
                                                        p(e_j), p(e_e), s)
                assert run_exp() == 0, lib.r2ik_last_error()
                torch.cuda.synchronize()
                ok = same(j.reshape(-1, 7), e_j) and same(el.reshape(-1, 3), e_e)
                if not no_limits:
                    ok = ok and same(state.repeat_interleave(K), e_state) and same(itv.repeat_interleave(K, dim=0), e_itv)
                else:
                    ok = ok and bool((proj.reshape(-1) == e_proj).all().item())
                t_sw = timed(run_sweep)
                t_ex = timed(run_exp)
                r = {"N": n, "K": K, "no_limits": no_limits, "angles": mode, "sweep_ms": t_sw[0], "sweep_min_max": t_sw[1:],
                     "expanded_ms": t_ex[0], "expanded_min_max": t_ex[1:], "model_ms": model,
                     "k1_solve_only_ms": t_solve[0], "k1_full_ms": t_full[0], "speedup_vs_expanded": t_ex[0] / t_sw[0],
                     "sweep_over_model": t_sw[0] / model, "reachable": float((state == 0).float().mean().item()),
                     "bit_identical": ok}
                rows.append(r)
                print(json.dumps(r), flush=True)
                assert ok, r
        del Pe, e_state, e_itv, e_j, e_e, e_proj
        torch.cuda.empty_cache()
    print(f"\n{header['card_name_power_limit']}  lib={header['lib']}")
    print(f"{'N':>8} {'K':>5} {'nl':>2} {'angles':>7} {'sweep ms':>9} {'expanded':>9} {'model':>9} {'x exp':>6} {'/model':>6}")
    for r in rows:
        print(f"{r['N']:>8} {r['K']:>5} {r['no_limits']:>2} {r['angles']:>7} {r['sweep_ms']:>9.4f} {r['expanded_ms']:>9.4f} "
              f"{r['model_ms']:>9.4f} {r['speedup_vs_expanded']:>6.2f} {r['sweep_over_model']:>6.2f}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"header": header, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
