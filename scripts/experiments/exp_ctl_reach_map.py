"""The controller's workspace map (r2ik_ctl_reach_map_u32) against its yardsticks.

For each grid (64^3 x 128, 128^3 x 512, 256^3 x 512 orientations over the reach cube, Fibonacci orientations), in one
process:
  ctl_map      r2ik_ctl_reach_map_u32, accepted + reachable volumes, for both arms, the standard and the DVT controller
               (singularity_offset -1.01 / 0.03) and nb_search_points K = 20 and 360
  symik_map    SymbolicIK.reach_map's entries on the same grid: r2ik_reach_map_u32 (mixed precision) and
               r2ik_reach_map_f64_u32 (all FP64) -- the cost of reachability alone
  materialised at 64^3 x 128 only: what a user has to do without the map -- build the 33.5 M poses [R_o | p_v] on the
               device, run the compacted discrete entry (r2ik_ctl_discrete_compact_f64) and sum the flags per voxel;
               its counts are checked against the map's
Kernel times are CUDA-event medians of `--rounds` windows of `--reps` launches after `--warmup` launches.

    python scripts/experiments/exp_ctl_reach_map.py [--lib path/to/libr2ik.so] [--quick] [--out prefix]
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

GRIDS = [(64, 128), (128, 512), (256, 512)]


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
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="256^3 x 512, r_arm, K = 20 only (launch-bounds variants)")
    ap.add_argument("--out", default=None, help="write <out>.json and <out>.txt")
    a = ap.parse_args()

    from reachy2_symbolic_ik_b200 import _native, build

    if a.lib:
        _native.use_library(a.lib)
    else:
        build.build()
    import torch

    from reachy2_symbolic_ik_b200 import ControlIK, fk, workspace

    header = {"card_name_power_limit": card(), "lib": a.lib or "in-tree", "warmup": a.warmup, "reps": a.reps,
              "rounds": a.rounds}
    print(json.dumps(header), flush=True)
    ctls = {False: ControlIK(urdf_path="../config_files/reachy2.urdf"),
            True: ControlIK(urdf_path="../config_files/reachy2.urdf", is_dvt=True)}
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    p = lambda t: C.c_void_p(None if t is None else t.data_ptr())   # noqa: E731
    i32 = C.c_int32

    def timed(fn):
        for _ in range(a.warmup):
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

    rows = []
    grids = [(256, 512)] if a.quick else GRIDS
    arms = ("r_arm",) if a.quick else ("r_arm", "l_arm")
    for n, n_ori in grids:
        eul = fk.fibonacci_orientations(n_ori)
        R = workspace.rpy_matrices(eul)
        for arm in arms:
            for dvt in ((False,) if a.quick else (False, True)):
                ctl = ctls[dvt]
                sv = ctl.symbolic_ik_solver[arm]
                lib, h = sv._handle.lib, sv._handle.h
                s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                origin, step, dims = workspace.reach_grid(sv.shoulder_position, sv.max_arm_length, n)
                origin, step = np.ascontiguousarray(origin), np.ascontiguousarray(step)
                dims = np.ascontiguousarray(dims, dtype=np.int32)
                ori = torch.from_numpy(R.reshape(-1, 9)).cuda()
                ori_e = torch.from_numpy(np.ascontiguousarray(eul)).cuda()
                acc = torch.empty((n, n, n), dtype=torch.int32, device="cuda")
                rea = torch.empty_like(acc)
                live = None
                for K in ((20,) if a.quick else (20, 360)):
                    ctl.nb_search_points = K
                    par = ctl._ctl_params(arm, "unconstrained", -4 * np.pi / 6, 0.01)

                    def run_map():
                        return lib.r2ik_ctl_reach_map_u32(h, C.byref(par), origin.ctypes.data_as(dp), step.ctypes.data_as(dp),
                                                          dims.ctypes.data_as(ip), p(ori), i32(0), i32(n_ori), p(acc), p(rea), s)

                    assert run_map() == 0, lib.r2ik_last_error()
                    t = timed(run_map)
                    r = {"what": "ctl_map", "n": n, "n_ori": n_ori, "arm": arm, "dvt": dvt, "K": K, "ms": t[0],
                         "min_max": t[1:], "pairs": n ** 3 * n_ori, "accepted": int(acc.sum()), "reachable": int(rea.sum())}
                    r["accepted_over_reachable"] = r["accepted"] / max(r["reachable"], 1)
                    live = int((rea > 0).sum())
                    rows.append(r)
                    print(json.dumps(r), flush=True)
                    if n == 64 and K == 20 and not a.quick:
                        rows.append(materialised(ctl, arm, dvt, origin, step, R, acc, timed))
                        print(json.dumps(rows[-1]), flush=True)
                ctl.nb_search_points = 20
                if not dvt:
                    sym = torch.empty_like(acc)
                    for entry in ("r2ik_reach_map_u32", "r2ik_reach_map_f64_u32"):
                        fn = getattr(lib, entry)

                        def run_sym():
                            return fn(h, origin.ctypes.data_as(dp), step.ctypes.data_as(dp), dims.ctypes.data_as(ip), p(ori_e),
                                      i32(0), i32(n_ori), p(sym), s)

                        assert run_sym() == 0, lib.r2ik_last_error()
                        t = timed(run_sym)
                        r = {"what": "symik_map_" + ("fp64" if "f64" in entry else "mixed"), "n": n, "n_ori": n_ori, "arm": arm,
                             "ms": t[0], "min_max": t[1:], "reachable": int(sym.sum()), "live_voxels": live}
                        rows.append(r)
                        print(json.dumps(r), flush=True)
                del acc, rea, ori, ori_e
                torch.cuda.empty_cache()

    lines = [f"{header['card_name_power_limit']}  lib={header['lib']}  warmup={a.warmup} reps={a.reps} rounds={a.rounds}",
             f"{'what':>20} {'grid':>12} {'arm':>5} {'ctl':>4} {'K':>4} {'ms':>9} {'min..max':>17} {'ns/pair':>8} "
             f"{'accepted':>11} {'reachable':>11} {'acc/reach':>9}"]
    for r in rows:
        grid = f"{r['n']}^3x{r['n_ori']}"
        ctl_s = ("dvt" if r.get("dvt") else "std") if "dvt" in r else ""
        lines.append(f"{r['what']:>20} {grid:>12} {r['arm']:>5} {ctl_s:>4} {r.get('K', ''):>4} {r['ms']:>9.3f} "
                     f"{r['min_max'][0]:>8.3f}..{r['min_max'][1]:<8.3f} {1e6 * r['ms'] / (r['n'] ** 3 * r['n_ori']):>8.4f} "
                     f"{r.get('accepted', ''):>11} {r.get('reachable', ''):>11} "
                     f"{format(r['accepted_over_reachable'], '.3f') if 'accepted_over_reachable' in r else '':>9}")
    txt = "\n".join(lines)
    print("\n" + txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out + ".json", "w") as f:
            json.dump({"header": header, "rows": rows}, f, indent=1)
        with open(a.out + ".txt", "w") as f:
            f.write(txt + "\n")


def materialised(ctl, arm, dvt, origin, step, R, acc, timed):
    """Without the map: build the n^3 x n_ori poses on the device, the compacted discrete entry, the per-voxel sum.  The
    voxel centres are computed on the host (262 144 x 3 doubles, a multiply then an add as the kernel does) and uploaded
    inside the timed window; the poses are written by broadcasting copies, so their bits equal the map's."""
    import torch

    n, n_ori = acc.shape[0], len(R)
    nv = n ** 3
    ix, iy, iz = np.meshgrid(*(np.arange(n) for _ in range(3)), indexing="ij")
    idx = np.stack([ix, iy, iz], axis=-1).reshape(-1, 3).astype(np.float64)
    Rd = torch.from_numpy(np.ascontiguousarray(R)).cuda()
    M = torch.empty((nv, n_ori, 4, 4), dtype=torch.float64, device="cuda")
    out = {}

    def run():
        P = torch.from_numpy(origin + idx * step).cuda(non_blocking=False)
        M[:, :, :3, :3] = Rd[None]
        M[:, :, :3, 3] = P[:, None, :]
        M[:, :, 3, :3] = 0.0
        M[:, :, 3, 3] = 1.0
        res = ctl.symbolic_inverse_kinematics_batch(arm, M.view(nv * n_ori, 4, 4), "discrete", compact=True,
                                                    out=out.get("res"))
        out["res"] = res
        out["counts"] = res[1].view(nv, n_ori).sum(dim=1, dtype=torch.int32)

    t = timed(run)
    equal = bool(torch.equal(out["counts"].view(n, n, n), acc))
    r = {"what": "materialised_discrete", "n": n, "n_ori": n_ori, "arm": arm, "dvt": dvt,
         "K": ctl.nb_search_points, "ms": t[0], "min_max": t[1:], "pairs": nv * n_ori, "accepted": int(out["counts"].sum()),
         "counts_equal_map": equal}
    del M, out
    torch.cuda.empty_cache()
    return r


if __name__ == "__main__":
    main()
