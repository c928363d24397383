"""Continuous mode of the kernel source on the host (tests/hostsim: the serial recursion of k_ctl_continuous and the phased
form of the k_cont_* kernels) on the trajectory families of continuous_edge_inputs.py, against the CPU oracle.  The GPU twin
is test_gpu_continuous_edges.py.

Every family runs at the SHAPES of continuous_edge_inputs.py (W around the 127 / 128 block edge, the 128-waypoint code tile,
the 8-waypoint theta tile and W % 8; T around the 64-trajectory blocks), as prefixes of one T_MAX x W_MAX batch."""
import numpy as np
import pytest

import continuous_edge_inputs as CE
from test_hostsim_parity import ARMS, cfg_for, ctl_params, hs, hs_continuous, urdf_params  # noqa: F401 (hs: fixture)

FAMILIES = [*CE.live_families("r_arm", 1, 2), "events"]


def _host(hs, oracle, arm):
    cfg, par = cfg_for(arm, urdf_params(), -1.01), ctl_params(oracle, arm)
    return lambda M, states=None, **kw: hs_continuous(hs, oracle, cfg, par, arm, M, states=states, **kw)  # noqa: E731


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("name", FAMILIES)
def test_family_vs_oracle(hs, oracle, arm, name):
    """Serial and phased forms against the oracle at every shape; phased (also with every 1st / 7th waypoint sent down the
    serial get_joints route) against serial; a run resumed at SPLITS equal to the one-shot run."""
    M, want, ill = CE.reference(oracle, arm, name)
    ocfg, opar = CE.oracle_config(oracle, arm)
    run = _host(hs, oracle, arm)
    worst = 0.0
    for T, W in CE.SHAPES:
        X = np.ascontiguousarray(M[:T, :W])
        w = oracle.ctl_continuous_batch(ocfg, opar, X)
        serial = run(X)
        worst = max(worst, CE.compare_with_oracle(f"{name} {arm} {T}x{W} serial", serial, w, ill[:T, :W]))
        for force in (0, 1, 7):
            CE.assert_same_trajectories(run(X, phased=True, force_serial=force), serial, f"{name} {arm} {T}x{W} phased force={force}")
    cuts = [c for c in CE.SPLITS if c < M.shape[1]]
    one = run(M)
    CE.assert_same_trajectories(CE.split_run(run, M, cuts), one, f"{name} {arm} split serial", atol=0)
    one_p = run(M, phased=True)
    CE.assert_same_trajectories(CE.split_run(lambda m, st: run(m, st, phased=True), M, cuts), one_p, f"{name} {arm} split phased")
    latched = float(want[3]["emergency_stop"].astype(bool).mean())
    max_ill = CE.MAX_ILL.get(name, CE.MAX_ILL_DEFAULT)
    print(f"[host continuous edges {name} {arm}] {M.shape[0]} x {M.shape[1]} waypoints: latched {int(want[3]['emergency_stop'].sum())}"
          f"/{M.shape[0]} trajectories, ill-conditioned {ill.mean():.4f}, max|err| well-conditioned {worst:.2e}")
    if name != "events":
        assert latched <= CE.LIVE_MAX_LATCHED.get(name, 0.0), f"{name}: {latched:.3f} of the trajectories latched"
    assert ill.mean() <= max_ill, f"{name}: ill-conditioned share {ill.mean():.4f} > {max_ill}"


@pytest.mark.parametrize("arm", ARMS)
def test_events_unfreeze(hs, oracle, arm):
    """Each trajectory of the event family resumed with "unfreeze" right after its event (an invalid rotation, a latching
    half turn or an edge_inputs pose at a block / tile edge): both forms against the oracle's segments."""
    M, want_all, _ = CE.reference(oracle, arm, "events")
    at = CE.event_families(arm)[1]
    run = _host(hs, oracle, arm)
    for t, want, ill in CE.unfreeze_references(oracle, arm):
        for phased in (False, True):
            got = CE.unfreeze_run(lambda m, st: run(m, st, phased=phased), oracle, M[t], at[t])
            CE.compare_with_oracle(f"events {arm} traj {t} ({CE.event_kind(t)}) unfreeze phased={phased}", got, want, ill)
    latched = want_all[3]["emergency_stop"].astype(bool)
    assert latched.mean() >= 0.5, f"only {int(latched.sum())} trajectories latched at their event"


@pytest.mark.parametrize("arm", ARMS)
def test_elbow_circle_normal_in_isclose_band(hs, oracle, arm):
    """Regression: an elbow-circle normal within the 1e-8 isclose band of +-e_x (the even trajectories of slow_rmfv), solved
    pose by pose.  rotation_matrix_from_vector then returns e_y, +-e_z, which are up to 1e-8 rad off the plane of the
    circle; the solver's fast interval route assumed an orthonormal frame and put the interval up to 1.6e-8 rad off the
    reference's until such poses went to the literal route."""
    from test_hostsim_parity import symik_vs_oracle

    M = CE.live_families(arm, only=("slow_rmfv",))["slow_rmfv"][::2].reshape(-1, 4, 4)
    ocfg = CE.oracle_config(oracle, arm)[0]
    rep, state, want = symik_vs_oracle(hs, oracle, f"hostsim rmfv band {arm}", cfg_for(arm, urdf_params(), -1.01), ocfg, M)
    rep.check(max_ill_fraction=0.0)
    assert (state == 0).mean() > 0.3
