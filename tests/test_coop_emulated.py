"""CPU: the COOPERATIVE tier (several CTAs per LP, simplex_cta.cuh "Cooperative tier") driven through the multi-CTA
fiber emulator against the oracle: group barriers, fused update + FTRAN, double-buffered inverse, blocked
Gauss-Jordan inversion with (emulated) DMMA tiles, leader-only Bland / polish / repair paths. Also pins the
decision-level tools of tests/parity_tools.py on the forced-path fixtures."""
import os

import numpy as np
import pytest

import emu_harness as E
import oracle
from parity_tools import classify_divergence, first_divergence
from problems import feasible_bounded_lp, knapsack, node_lp, raw_lp, standard_form

HERE = os.path.dirname(os.path.abspath(__file__))


def _close(a, b, tol=1e-9):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b))) <= tol


@pytest.mark.parametrize("m,n,count,G,groups,T", [(5, 12, 4, 2, 1, 32), (12, 30, 6, 3, 2, 64), (40, 90, 2, 4, 1, 64),
                                                  (33, 70, 2, 5, 1, 32), (20, 50, 2, 25, 1, 32), (20, 50, 2, 1, 2, 64)])
def test_coop_tier_matches_oracle(m, n, count, G, groups, T):
    rng = np.random.default_rng(100 * m + n)
    c, A, b = feasible_bounded_lp(rng, m, n, count)
    g = E.coop_batch(c, A, b, T=T, G=G, groups=groups, trace_cap=256)
    o = oracle.simplex_batch(c, A, b)
    assert (g["status"] == o["status"]).all() and (o["status"] == 0).all()
    assert _close(g["optF"], o["optF"]) and _close(g["x"], o["x"])
    assert (g["stats"][:, 3] >= 1).all()  # dense start: the blocked (DMMA) inversion ran
    o0 = oracle.simplex(c[0], A[0], b[0], trace_cap=256)
    k = first_divergence(o0.trace, g["trace"][g["trace"][:, 0] >= 0])
    if k >= 0:  # only a near-tie may separate the pivot sequences
        why = classify_divergence(c[0], A[0], b[0], o0.trace, g["trace"][g["trace"][:, 0] >= 0], k,
                                  oracle.initial_basis(A[0]), o0.basis)
        assert why != "REAL", why


def test_coop_tier_refactor_and_shuffled_schedule():
    rng = np.random.default_rng(5)
    c, A, b = feasible_bounded_lp(rng, 20, 50, 3)
    o = oracle.simplex_batch(c, A, b)
    for G, T, rp, sh in [(3, 64, 5, True), (7, 32, 3, False)]:
        g = E.coop_batch(c, A, b, T=T, G=G, refactor_period=rp, shuffle_order=sh)
        assert (g["status"] == 0).all() and _close(g["optF"], o["optF"]) and _close(g["x"], o["x"])
        assert (g["stats"][:, 3] > 2).all()  # periodic re-inversion through the group


def test_coop_tier_status_parity_on_raw_lps():
    rng = np.random.default_rng(11)
    for (m, n, count, pz) in [(3, 7, 40, 0.0), (6, 10, 40, 0.3), (5, 5, 8, 0.0), (6, 4, 4, 0.0)]:
        c, A, b = raw_lp(rng, m, n, count, pz)
        g = E.coop_batch(c, A, b, T=32, G=3, groups=2)
        o = oracle.simplex_batch(c, A, b, max_pivots=20000)
        assert (g["status"] == o["status"]).sum() >= count - 1
        ok = (g["status"] == 0) & (o["status"] == 0)
        if ok.any():
            assert _close(g["optF"][ok], o["optF"][ok]) and _close(g["x"][ok], o["x"][ok])


def test_coop_tier_wave_of_knapsack_children():
    rng = np.random.default_rng(3)
    p = knapsack(rng, 10, 3)
    c0, A0, b0 = standard_form(p)
    L, nodes = 2, 6
    bvar = rng.integers(0, 10, size=(nodes, L)).astype(np.int32)
    bsign = rng.choice([-1.0, 1.0], size=(nodes, L))
    brhs = np.where(bsign > 0, 0.0, -1.0)
    g = E.coop_batch(c0, A0, b0, bvar=bvar, bsign=bsign, brhs=brhs, shared_root=True, T=32, G=3, groups=2)
    for k in range(nodes):
        c, A, b = node_lp(c0, A0, b0, bvar[k], bsign[k], brhs[k])
        o = oracle.simplex(c, A, b)
        assert g["status"][k] == o.status
        if o.status == 0:
            assert _close(g["optF"][k], o.optF) and _close(g["x"][k], o.x[: A0.shape[1]])


def test_forced_paths_fire_and_divergences_are_near_ties():
    """forced_paths.npz: LPs on which the ORACLE runs replaceBland, the artificial-still-basic repair loop, or
    rejects columns in the basis scan. The kernel must reach the same status / objective, must run the same machinery
    (Bland / basis-scan counters), and wherever its pivot sequence leaves the oracle's the two choices must be a
    near-tie in the quantity floats.MinIdx compared."""
    z = np.load(os.path.join(HERE, "golden", "forced_paths.npz"))
    fired = {"bland": 0, "repair": 0, "scan": 0}
    why_all = []
    for kind in ("bland", "repair", "scan"):
        for k in range(int(z[kind + "_count"])):
            c, A, b = z[f"{kind}{k}_c"], z[f"{kind}{k}_A"], z[f"{kind}{k}_b"]
            for coop in (False, True):
                if coop:
                    g = E.coop_batch(c[None], A[None], b[None], T=32, G=3, trace_cap=256)
                else:
                    g = E.simplex_batch(c[None], A[None], b[None], T=64)
                s = g["stats"][0]
                assert g["status"][0] == int(z[f"{kind}{k}_status"])
                assert abs(g["optF"][0] - float(z[f"{kind}{k}_z"])) <= 1e-9 * max(1.0, abs(float(z[f"{kind}{k}_z"])))
                if kind == "scan":
                    assert s[5] == 1  # the optimistic last-m block was refused, the reverse scan ran
                    st = oracle.initial_basis(A)
                if coop:
                    fired["bland"] += int(s[2] > 0)
                    fired["repair"] += int(s[6] > 0)
                    fired["scan"] += int(s[5] > 0)
                    tr_ref = z[f"{kind}{k}_trace"]
                    tr = g["trace"][g["trace"][:, 0] >= 0]
                    d = first_divergence(tr_ref, tr)
                    if d >= 0:
                        why = classify_divergence(c, A, b, tr_ref, tr, d, oracle.initial_basis(A), z[f"{kind}{k}_basis"])
                        why_all.append(why)
                        assert why != "REAL", (kind, k, d, why)
    print("paths fired (of 18 LPs):", fired, "divergences:", {w: why_all.count(w) for w in set(why_all)})
    assert fired["bland"] >= 4 and fired["repair"] >= 3 and fired["scan"] >= 6


def test_robust_mode_stops_at_a_pivot_cap_the_caller_set():
    """gm_options.robust (opt-in, no reference counterpart): an LP the first pass cannot finish is solved again with
    its Phase II on a perturbed vertex and the basis found re-evaluated on the true right-hand side. A pivot cap the
    caller sets is a total over all passes: robust mode stops at it like the plain solve, on every kind of tier, at the
    same vertex; with the default cap every LP reaches the oracle's optimum."""
    rng = np.random.default_rng(4)
    c, A, b = feasible_bounded_lp(rng, 12, 30, 4)
    o = oracle.simplex_batch(c, A, b)
    plain = E.simplex_batch(c, A, b, max_pivots=5, T=64)
    assert (plain["status"] == 68).all()                                   # without the option: the cap is reported
    E.set_robust(True)
    try:
        capped = [E.simplex_batch(c, A, b, max_pivots=5, T=64), E.simplex_batch(c, A, b, max_pivots=5, T=256, reg=True),
                  E.coop_batch(c, A, b, T=32, G=3, max_pivots=5)]
        full = [E.simplex_batch(c, A, b, T=64), E.simplex_batch(c, A, b, T=256, reg=True), E.coop_batch(c, A, b, T=32, G=3)]
    finally:
        E.set_robust(False)
    for g in capped:
        assert (g["status"] == 68).all() and not (g["stats"][:, 5] & 2).any()  # bit 1: no robust pass ran
        assert (g["stats"][:, 0] + g["stats"][:, 1] == 5).all()
        assert _close(g["x"], plain["x"])
    for g in full:
        assert (g["status"] == 0).all() and _close(g["optF"], o["optF"]) and _close(g["x"], o["x"])


def test_degenerate_lp_that_stalls_some_gpu_schedules():
    """tests/golden/degenerate_105x137.npz: the LP (n barely above m, a degenerate optimal vertex) on which tier 6 with
    1 - 5 CTAs stalls at the optimal vertex on the GPU while tiers 3 / 5 and 37 CTAs do not (DESIGN.md §3). The oracle
    and the emulated cooperative tier both get through it on Bland calls; they must agree on the optimum."""
    z = np.load(os.path.join(HERE, "golden", "degenerate_105x137.npz"))
    c, A, b = z["c"], z["A"], z["b"]
    o = oracle.simplex(c[0], A[0], b[0])
    assert o.status == 0 and o.bland_calls > 50
    g = E.coop_batch(c, A, b, T=64, G=2)
    assert g["status"][0] == 0 and g["stats"][0, 2] > 50
    assert _close(g["optF"][0], o.optF) and _close(g["x"][0], o.x)
