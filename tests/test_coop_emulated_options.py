"""CPU: the caller-facing options of the C ABI on the emulated COOPERATIVE tier (several CTAs per LP, groups of
emulated CTAs scheduled in shuffled order): `tol`, `initialBasic`, refactor_period = 1, the pivot cap, and early
exits mixed with healthy LPs in one batch, against the CPU oracle and the extended-precision certificate of
test_gpu_solver_options. A leader that leaves its helpers behind on an early exit shows here as "barrier divergence"."""
import numpy as np
import pytest

import emu_harness as E
import oracle
from gomilp_b200 import status as S
from problems import feasible_bounded_lp
from test_gpu_solver_options import (EXIT_STATUS, RTOL, basis_cases, check_certificate, mixed_batch, rel, same_bases,
                                     slack_batch)

GROUPS = [2, 3]


def coop(c, A, b, G, groups=2, **kw):
    return E.coop_batch(c, A, b, T=32, G=G, groups=groups, shuffle_order=True, **kw)


@pytest.mark.parametrize("G", GROUPS)
def test_emulated_coop_tol(G):
    m, n, count = 20, 50, 8
    c, A, b = feasible_bounded_lp(np.random.default_rng(60 + G), m, n, count)
    g0 = coop(c, A, b, G)
    o0 = oracle.simplex_batch(c, A, b)
    worst = 0.0
    for tol in (1e-9, 1e-6, 1e-3, 0.1):
        g = coop(c, A, b, G, tol=tol)
        o = oracle.simplex_batch(c, A, b, tol=tol)
        assert (g["status"] == o["status"]).all() and (g["status"] == S.GM_OK).all()
        for k in range(count):
            worst = max(worst, check_certificate(c[k], A[k], b[k], g["basis"][k], g["x"][k], tol))
        piv = g["stats"][:, 0] + g["stats"][:, 1]
        assert (piv <= g0["stats"][:, 0] + g0["stats"][:, 1]).all()
        same = same_bases(g, o)
        assert same.mean() >= 0.9
        assert rel(g["optF"][same], o["optF"][same]) <= RTOL and rel(g["x"][same], o["x"][same]) <= RTOL
        if tol == 0.1:
            early = g["optF"] > o0["optF"] + RTOL * np.maximum(1.0, np.abs(o0["optF"]))
            assert early.mean() >= 0.3
    print(f"emulated tier 6 G={G}, tol: largest deviation of x from the certificate {worst:.1e}")


@pytest.mark.parametrize("G", GROUPS)
def test_emulated_coop_initial_basic(G):
    """Every initialBasic case, each followed in the same batch by a healthy LP started from a feasible basis, so a
    group that an early exit left in a bad state is noticed on the next LP it takes."""
    m, n = 16, 40
    rng = np.random.default_rng(70 + G)
    c, A, b = feasible_bounded_lp(rng, m, n)
    cases = basis_cases(c, A, b, rng)
    start = dict((name, ib) for name, ib, _, _ in cases)["feasible"]
    cs, As, bs, ibs = [], [], [], []
    for _, ib, (cc, AA, bb), _ in cases:
        cs += [cc, c]
        As += [AA, A]
        bs += [bb, b]
        ibs += [ib, start]
    g = coop(np.array(cs), np.array(As), np.array(bs), G, initial_basic=np.array(ibs))
    healthy = oracle.simplex(c, A, b, initial_basic=start)
    for q, (name, ib, (cc, AA, bb), want) in enumerate(cases):
        k = 2 * q
        if want is not None:
            assert g["status"][k] == want, (name, g["status"][k])
            assert g["stats"][k, 7] == 0
        else:
            o = oracle.simplex(cc, AA, bb, initial_basic=ib)
            assert g["status"][k] == o.status == S.GM_OK, name
            assert rel(g["x"][k], o.x) <= RTOL and rel(g["optF"][k], o.optF) <= RTOL, name
            check_certificate(cc, AA, bb, g["basis"][k], g["x"][k])
            if name == "optimal":
                assert g["stats"][k, 0] + g["stats"][k, 1] == 0
        assert g["status"][k + 1] == S.GM_OK, name
        assert rel(g["x"][k + 1], healthy.x) <= RTOL and rel(g["optF"][k + 1], healthy.optF) <= RTOL, name


@pytest.mark.parametrize("G", GROUPS)
@pytest.mark.parametrize("count,groups", [(14, 2), (6, 8)])
def test_emulated_coop_early_exits_in_mixed_batches(G, count, groups):
    m, n = 16, 42
    c, A, b, kinds = mixed_batch(m, n, count, 900 + count)
    g = coop(c, A, b, G, groups=groups)
    o = oracle.simplex_batch(c, A, b)
    assert (g["status"] == o["status"]).all(), list(zip(kinds, g["status"], o["status"]))
    for k, kind in enumerate(kinds):
        if kind in EXIT_STATUS:
            assert g["status"][k] == EXIT_STATUS[kind], kind
    ok = np.array([k is None for k in kinds])
    assert (g["status"][ok] == S.GM_OK).all()
    assert rel(g["optF"][ok], o["optF"][ok]) <= RTOL and rel(g["x"][ok], o["x"][ok]) <= RTOL
    alone = coop(c[ok], A[ok], b[ok], G, groups=groups)
    for key in ("status", "optF", "x", "basis", "stats"):
        assert np.array_equal(alone[key], g[key][ok]), key


@pytest.mark.parametrize("G", GROUPS)
def test_emulated_coop_refactor_every_pivot(G):
    m, n, count = 20, 50, 4
    c, A, b = feasible_bounded_lp(np.random.default_rng(80 + G), m, n, count)
    o = oracle.simplex_batch(c, A, b)
    base = coop(c, A, b, G)
    g = coop(c, A, b, G, refactor_period=1)
    piv = g["stats"][:, 0] + g["stats"][:, 1]
    assert (g["status"] == o["status"]).all() and (g["status"] == S.GM_OK).all()
    assert rel(g["optF"], o["optF"]) <= RTOL and rel(g["x"], o["x"]) <= RTOL
    assert (g["stats"][:, 3] >= piv).all()
    assert np.mean([set(g["basis"][i]) == set(base["basis"][i]) for i in range(count)]) >= 0.9
    assert np.mean(piv == base["stats"][:, 0] + base["stats"][:, 1]) >= 0.9


@pytest.mark.parametrize("G", GROUPS)
def test_emulated_coop_pivot_cap(G):
    """Slack-form data: no Phase I, so the oracle's per-call cap and the engine's total cap coincide."""
    m, n, count = 16, 40, 4
    c, A, b = slack_batch(m, n, count, 90 + G)
    for k in (1, 2, 7, 40):
        g = coop(c, A, b, G, max_pivots=k)
        o = oracle.simplex_batch(c, A, b, max_pivots=k)
        piv = g["stats"][:, 0] + g["stats"][:, 1]
        assert (g["stats"][:, 4] == 0).all() and (g["status"] == o["status"]).all(), k
        capped = g["status"] == S.GM_ERR_ITERATION_LIMIT
        assert (piv[capped] == k).all() and (piv <= k).all()
        assert rel(g["x"], o["x"]) <= RTOL and rel(g["optF"], o["optF"]) <= RTOL, k
