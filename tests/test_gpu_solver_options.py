"""GPU (-m gpu): the parts of the C ABI that GoMILP's own branch-and-bound never passes, on every tier: `tol`,
`initialBasic`, gm_options.max_pivots, gm_options.refactor_period, the device-buffer entry point, early exits inside
mixed batches, and run-to-run reproducibility of tiers 5 and 6.

Two references: the CPU oracle (status, objective and x at 1e-9 relative), and `certificate()`, which rebuilds the
vertex and the reduced costs of the basis the kernel reports in extended precision, so that the stop rule
`min r >= -tol` is checked whatever pivot path the kernel took. The largest deviation from the certificate seen on
each tier is printed at the end of every test that computes one."""
from functools import lru_cache

import numpy as np
import pytest

import gomilp_b200 as gm
import oracle
from gomilp_b200 import status as S
from problems import feasible_bounded_lp

pytestmark = pytest.mark.gpu
RTOL = 1e-9
SMALL, LARGE = (48, 110), (120, 250)
# (shape, forced tier, CTAs per LP in tier 6); tier 0 = the shape's own choice. Tier 2 keeps W and the basis
# inverse in shared memory, (m n + m^2) doubles: 120 x 250 does not fit in 227 KB and runs on tiers 3-6.
TIERS = ([(SMALL, t, 0) for t in (1, 2, 3, 4, 5)] + [(SMALL, 6, G) for G in (1, 3, 37)] + [(SMALL, 0, 0)] +
         [(LARGE, t, 0) for t in (3, 4, 5)] + [(LARGE, 6, G) for G in (1, 3, 37)] + [(LARGE, 0, 0)])
TIER_IDS = [f"{m}x{n}-{'auto' if t == 0 else f'tier{t}'}{f'-G{G}' if G else ''}" for (m, n), t, G in TIERS]
EXIT_KINDS = ("zero_row_b", "zero_row", "zero_col_neg", "zero_col", "phase1_infeasible", "unbounded", "dup_row")
EXIT_STATUS = {"zero_row_b": S.GM_ERR_INFEASIBLE, "zero_row": S.GM_ERR_ZERO_ROW, "zero_col_neg": S.GM_ERR_UNBOUNDED,
               "zero_col": S.GM_ERR_ZERO_COLUMN}


def rel(a, b) -> float:
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) if a.size else 0.0


def certificate(c, A, b, basis):
    """Vertex, duals, reduced costs and cond1(B) of `basis`: B x_B = b and B'y = c_B solved in float64, then one
    step of iterative refinement with the residuals in long double. r = c - A'y is returned in long double."""
    L = np.longdouble
    basis = np.asarray(basis, dtype=np.int64)
    B = A[:, basis]
    BL = B.astype(L)
    xB = np.linalg.solve(B, b)
    xB = xB + np.linalg.solve(B, (b.astype(L) - BL @ xB.astype(L)).astype(float))
    cB = c[basis]
    y = np.linalg.solve(B.T, cB)
    y = y + np.linalg.solve(B.T, (cB.astype(L) - BL.T @ y.astype(L)).astype(float))
    x = np.zeros(A.shape[1])
    x[basis] = xB
    r = c.astype(L) - A.astype(L).T @ y.astype(L)
    return x, y, r, np.linalg.cond(B, 1)


def check_certificate(c, A, b, basis, x, tol=0.0) -> float:
    """The kernel's x is the vertex of its basis, that vertex is feasible, and the stop rule held there."""
    xc, _, r, cond = certificate(c, A, b, basis)
    assert cond < 1e12, cond
    assert xc[basis].min() >= -1e-9
    assert float(r.min()) >= -tol - 1e-9 * max(1.0, float(np.abs(c).max())), (float(r.min()), tol)
    dev = rel(x, xc)
    assert dev <= RTOL, dev
    return dev


class Worst:
    """Largest deviation from the certificate per tier label, printed as one line."""

    def __init__(self, what):
        self.what, self.v = what, {}

    def add(self, label, dev):
        self.v[label] = max(self.v.get(label, 0.0), dev)

    def report(self):
        print(f"{self.what}: largest deviation of x from the certificate " +
              ", ".join(f"{k} {v:.1e}" for k, v in sorted(self.v.items())))


def tier_label(tier, G=0):
    return f"tier {tier}" + (f" G={G}" if tier == 6 and G else "")


def solve(cfg_tier, G, c, A, b, tol=0.0, **opts):
    try:
        gm.set_options(force_tier=cfg_tier, coop_group=G, **opts)
        g = gm.simplex_batch(c, A, b, tol=tol)
        tier = gm.last_timing()["tier"]
    finally:
        gm.set_options()
    if cfg_tier:
        assert tier == cfg_tier
    g["tier"] = tier
    return g


@lru_cache(maxsize=None)
def batch(m, n, count, seed):
    return feasible_bounded_lp(np.random.default_rng(seed), m, n, count)


@lru_cache(maxsize=None)
def oracle_batch(m, n, count, seed, tol=0.0, max_pivots=0, kind="dense"):
    c, A, b = batch(m, n, count, seed) if kind == "dense" else slack_batch(m, n, count, seed)
    return oracle.simplex_batch(c, A, b, tol=tol, threads=oracle.num_hw_threads(), max_pivots=max_pivots)


@lru_cache(maxsize=None)
def slack_batch(m, n, count, seed):
    """[R I] x = b with b > 0: the slack basis is feasible, so neither the engine nor the oracle runs Phase I."""
    rng = np.random.default_rng(seed)
    A = np.zeros((count, m, n))
    A[:, :, : n - m] = rng.random((count, m, n - m))
    A[:, :, n - m:] = np.eye(m)
    b = 1.0 + rng.random((count, m))
    c = np.zeros((count, n))
    c[:, : n - m] = -rng.random((count, n - m))
    return c, A, b


def early_exit_lp(rng, m, n, kind):
    """A feasible bounded LP turned into one that exits early: a zero row with b != 0 / b = 0, a zero column with
    c < 0 / c >= 0, a Phase-I-infeasible row (positive row, negative b), an unbounded ray (x_{n-2} + x_{n-1} moves
    along a null direction of A at cost -1), or a duplicated row (rank-deficient A, consistent b)."""
    c, A, b = feasible_bounded_lp(rng, m, n)
    i, j = int(rng.integers(m)), int(rng.integers(n))
    if kind == "zero_row_b":
        A[i], b[i] = 0.0, 1.0
    elif kind == "zero_row":
        A[i], b[i] = 0.0, 0.0
    elif kind == "zero_col_neg":
        A[:, j], c[j] = 0.0, -1.0
    elif kind == "zero_col":
        A[:, j], c[j] = 0.0, 1.0
    elif kind == "phase1_infeasible":
        A[i], b[i] = np.abs(A[i]) + 0.1, -1.0
    elif kind == "unbounded":
        A[:, n - 1] = -A[:, n - 2]
        c[n - 1] = -c[n - 2] - 1.0
        b = A @ (rng.random(n) * (rng.random(n) < 0.5))
    elif kind == "dup_row":
        A[(i + 1) % m] = A[i]
        b = A @ (rng.random(n) * (rng.random(n) < 0.5))
    else:
        raise ValueError(kind)
    return c, A, b


@lru_cache(maxsize=None)
def mixed_batch(m, n, count, seed):
    """Even slots healthy LPs, odd slots the early exits in turn. Returns c, A, b, kinds (None = healthy)."""
    rng = np.random.default_rng(seed)
    cs, As, bs, kinds = [], [], [], []
    for k in range(count):
        kind = None if k % 2 == 0 else EXIT_KINDS[(k // 2) % len(EXIT_KINDS)]
        c, A, b = feasible_bounded_lp(rng, m, n) if kind is None else early_exit_lp(rng, m, n, kind)
        cs.append(c), As.append(A), bs.append(b), kinds.append(kind)
    return np.array(cs), np.array(As), np.array(bs), tuple(kinds)


@lru_cache(maxsize=None)
def oracle_mixed(m, n, count, seed):
    c, A, b, _ = mixed_batch(m, n, count, seed)
    return oracle.simplex_batch(c, A, b, threads=oracle.num_hw_threads())


def basis_cases(c, A, b, rng):
    """Initial bases for one feasible bounded LP: (name, basis, LP data, expected status or None = as the oracle).
    'feasible' is the optimal basis of another cost vector: feasible for (A, b), not optimal for c."""
    m, n = A.shape
    o = oracle.simplex(c, A, b)
    assert o.status == S.GM_OK
    y2 = rng.standard_normal(m)
    c2 = A.T @ y2 + rng.random(n)
    o2 = oracle.simplex(c2, A, b)
    assert o2.status == S.GM_OK
    for _ in range(200):
        bad = np.sort(rng.choice(n, m, replace=False))
        B = A[:, bad]
        if np.linalg.cond(B, 1) < 1e6 and np.linalg.solve(B, b).min() < -1e-3:
            break
    else:
        raise AssertionError("no infeasible basis found")
    dup = o.basis.copy()
    dup[1] = dup[0]
    Ad = A.copy()
    Ad[:, o.basis[1]] = Ad[:, o.basis[0]]  # two basic columns equal: a singular basis
    out_of_range = o.basis.copy()
    out_of_range[m // 2] = n
    return [("optimal", o.basis, (c, A, b), None), ("feasible", o2.basis, (c, A, b), None),
            ("infeasible", bad, (c, A, b), S.GM_PANIC_INITIAL_BASIC),
            ("duplicate", dup, (c, A, b), S.GM_PANIC_INITIAL_BASIC),
            ("dependent", o.basis, (c, Ad, b), S.GM_PANIC_INITIAL_BASIC),
            ("out_of_range", out_of_range, (c, A, b), S.GM_ERR_BAD_ARGUMENT)]


def same_bases(g, o):
    return np.array([set(g["basis"][i]) == set(o["basis"][i]) for i in range(len(g["basis"]))])


# ---- (a) tol ------------------------------------------------------------------------------------------------------

@pytest.mark.timeout(300)
@pytest.mark.parametrize("shape,tier,G", TIERS, ids=TIER_IDS)
def test_tol_stop_rule_on_every_tier(shape, tier, G):
    """Phase II stops at min r >= -tol. At tol = 0.1 most LPs stop at a vertex that is not optimal, so a tier that
    ignores tol reaches the true optimum and fails the oracle comparison."""
    m, n = shape
    count, seed = 16, 7 * m + n
    c, A, b = batch(m, n, count, seed)
    g0 = solve(tier, G, c, A, b)
    o0 = oracle_batch(m, n, count, seed)
    worst = Worst(f"tol {m}x{n} {tier_label(g0['tier'], G)}")
    for tol in (0.0, 1e-9, 1e-6, 1e-3, 0.1):
        g = solve(tier, G, c, A, b, tol=tol)
        o = oracle_batch(m, n, count, seed, tol=tol)
        assert (g["status"] == o["status"]).all() and (g["status"] == S.GM_OK).all(), tol
        for k in range(count):
            worst.add(f"tol={tol:g}", check_certificate(c[k], A[k], b[k], g["basis"][k], g["x"][k], tol))
        assert (g["pivots"] <= g0["pivots"]).all(), tol
        same = same_bases(g, o)
        assert rel(g["optF"][same], o["optF"][same]) <= RTOL and rel(g["x"][same], o["x"][same]) <= RTOL
        assert same.mean() >= 0.9, (tol, same.mean())
        if tol == 0.1:
            early = g["optF"] > o0["optF"] + RTOL * np.maximum(1.0, np.abs(o0["optF"]))
            print(f"tol 0.1: {early.sum()}/{count} LPs stop before the optimum")
            assert early.mean() >= 0.3
    worst.report()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("shape,tier,G", [(SMALL, 1, 0), (SMALL, 2, 0), (LARGE, 3, 0), (LARGE, 5, 0), (LARGE, 6, 3)],
                         ids=["48x110-tier1", "48x110-tier2", "120x250-tier3", "120x250-tier5", "120x250-tier6-G3"])
def test_tol_in_robust_mode(shape, tier, G):
    """Robust mode runs the warm-capable kernel variants; `tol` must reach them the same way."""
    m, n = shape
    count, seed = 16, 7 * m + n
    c, A, b = batch(m, n, count, seed)
    for tol in (1e-3, 0.1):
        plain = solve(tier, G, c, A, b, tol=tol)
        rob = solve(tier, G, c, A, b, tol=tol, robust=True)
        o = oracle_batch(m, n, count, seed, tol=tol)
        assert (rob["status"] == o["status"]).all()
        assert rel(rob["optF"], plain["optF"]) <= RTOL and rel(rob["x"], plain["x"]) <= RTOL
        assert (rob["pivots"] == plain["pivots"]).all() and not (rob["stats"][:, 5] & 2).any()
        for k in range(count):
            check_certificate(c[k], A[k], b[k], rob["basis"][k], rob["x"][k], tol)


# ---- (b) initialBasic ----------------------------------------------------------------------------------------------

def _simplex(tier, G, c, A, b, ib):
    try:
        gm.set_options(force_tier=tier, coop_group=G)
        try:
            r = gm.simplex(c, A, b, initial_basic=ib)
        except gm.EngineError as e:  # codes >= GM_ERR_BAD_SHAPE come back as exceptions from the binding
            r = gm.LPResult(e.code, float("nan"), None, None, 0)
        t = gm.last_timing()
    finally:
        gm.set_options()
    return r, t


def _initial_basic_cases(tier, G, c, A, b, rng, worst, label):
    healthy = oracle.simplex(c, A, b)
    for name, ib, (cc, AA, bb), want in basis_cases(c, A, b, rng):
        r, t = _simplex(tier, G, cc, AA, bb, ib)
        if tier:
            assert t["tier"] == tier, name
        if want is not None:
            assert r.status == want, (name, r.status)
            assert r.x is None
            # the group / CTA that returned early must solve the next LP cleanly
            h, _ = _simplex(tier, G, c, A, b, None)
            assert h.status == S.GM_OK and rel(h.x, healthy.x) <= RTOL and rel(h.optF, healthy.optF) <= RTOL, name
            continue
        o = oracle.simplex(cc, AA, bb, initial_basic=ib)
        assert r.status == o.status == S.GM_OK, (name, r.status, o.status)
        assert rel(r.x, o.x) <= RTOL and rel(r.optF, o.optF) <= RTOL, name
        worst.add(label, check_certificate(cc, AA, bb, r.basis, r.x))
        if name == "optimal":
            assert r.pivots == 0
        print(f"{label} {name}: {r.pivots} pivots (oracle {o.pivots})")


@pytest.mark.timeout(300)
@pytest.mark.parametrize("shape,tier,G", TIERS, ids=TIER_IDS)
def test_initial_basic_on_every_tier(shape, tier, G):
    m, n = shape
    rng = np.random.default_rng(31 * m + n)
    c, A, b = feasible_bounded_lp(rng, m, n)
    worst = Worst(f"initialBasic {m}x{n}")
    _initial_basic_cases(tier, G, c, A, b, rng, worst, tier_label(tier, G) if tier else "auto")
    worst.report()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("m", [100, 150, 300])
def test_initial_basic_on_the_automatic_cooperative_choice(m):
    """gm_simplex is a batch of one: for m >= 96 the engine puts min(m / 2, SMs) CTAs on it (tier 6)."""
    n = 2 * m + 10
    rng = np.random.default_rng(m)
    c, A, b = feasible_bounded_lp(rng, m, n)
    r, t = _simplex(0, 0, c, A, b, None)
    import torch
    assert t["tier"] == 6 and t["grid"] == min(m // 2, torch.cuda.get_device_properties(0).multi_processor_count), t
    worst = Worst(f"initialBasic {m}x{n} auto")
    _initial_basic_cases(0, 0, c, A, b, rng, worst, f"tier 6 G={t['grid']}")
    worst.report()


# ---- (c) max_pivots ------------------------------------------------------------------------------------------------

@pytest.mark.timeout(300)
@pytest.mark.parametrize("shape,tier,G", TIERS, ids=TIER_IDS)
def test_pivot_cap_on_every_tier(shape, tier, G):
    """The engine caps Phase I + Phase II pivots together; the oracle caps each of its simplex calls. On slack-form
    data neither runs Phase I and the two must agree on status and on the mid-path vertex; on dense data the
    engine's own contract is checked."""
    m, n = shape
    count, seed = 16, 3 * m + n
    cs, As, bs = slack_batch(m, n, count, seed)
    cd, Ad, bd = batch(m, n, count, seed)
    fired = 0
    for k in (1, 2, 7, 40):
        g = solve(tier, G, cs, As, bs, max_pivots=k)
        o = oracle_batch(m, n, count, seed, max_pivots=k, kind="slack")
        piv = g["stats"][:, 0] + g["stats"][:, 1]
        assert (g["stats"][:, 4] == 0).all()
        assert (g["status"] == o["status"]).all(), k
        capped = g["status"] == S.GM_ERR_ITERATION_LIMIT
        fired += int(capped.sum())
        assert (piv[capped] == k).all() and (piv <= k).all()
        assert rel(g["x"], o["x"]) <= RTOL and rel(g["optF"], o["optF"]) <= RTOL, k
        gd = solve(tier, G, cd, Ad, bd, max_pivots=k)
        pd = gd["stats"][:, 0] + gd["stats"][:, 1]
        assert (pd <= k).all() and (pd[gd["status"] == S.GM_ERR_ITERATION_LIMIT] == k).all()
        assert np.isin(gd["status"], [S.GM_OK, S.GM_ERR_ITERATION_LIMIT,
                                      S.GM_ERR_PHASE1_WRAPPED + S.GM_ERR_ITERATION_LIMIT]).all()
    assert fired >= count  # k = 1 stops every LP
    # robust mode may not lift a cap the caller set: it is a total over all passes
    for k in (2, 7):
        rob = solve(tier, G, cd, Ad, bd, max_pivots=k, robust=True)
        plain = solve(tier, G, cd, Ad, bd, max_pivots=k)
        pr = rob["stats"][:, 0] + rob["stats"][:, 1]
        assert (pr <= k).all(), (k, pr.max())
        assert (rob["status"] == plain["status"]).all() and not (rob["stats"][:, 5] & 2).any()
        assert (plain["status"] != S.GM_OK).sum() >= count // 2


# ---- (d) refactor_period -------------------------------------------------------------------------------------------

@pytest.mark.timeout(300)
@pytest.mark.parametrize("shape,tier,G", TIERS, ids=TIER_IDS)
def test_refactor_period_on_every_tier(shape, tier, G):
    """Period 1 rebuilds the basis inverse after every pivot (in tier 6: leader -> group inversion -> leader)."""
    m, n = shape
    count, seed = 12, 5 * m + n
    c, A, b = batch(m, n, count, seed)
    o = oracle_batch(m, n, count, seed)
    base = solve(tier, G, c, A, b)
    worst = Worst(f"refactor_period {m}x{n} {tier_label(base['tier'], G)}")
    for period in (1, 2, 5):
        g = solve(tier, G, c, A, b, refactor_period=period)
        assert (g["status"] == o["status"]).all() and (g["status"] == S.GM_OK).all()
        assert rel(g["optF"], o["optF"]) <= RTOL and rel(g["x"], o["x"]) <= RTOL, period
        assert (g["stats"][:, 3] >= g["pivots"] // period).all(), period
        same = np.mean([set(g["basis"][i]) == set(base["basis"][i]) for i in range(count)])
        assert same >= 0.9 and np.mean(g["pivots"] == base["pivots"]) >= 0.9, period
        for k in range(count):
            worst.add(f"period {period}", check_certificate(c[k], A[k], b[k], g["basis"][k], g["x"][k]))
    worst.report()


# ---- (e) gm_simplex_batch_device -----------------------------------------------------------------------------------

def _device_call(c, A, b, stream, with_basis=True, tol=0.0):
    import torch
    count, m, n = A.shape
    dev = torch.device("cuda", 0)
    out = {"status": torch.zeros(count, dtype=torch.int32, device=dev), "optF": torch.zeros(count, device=dev,
           dtype=torch.float64), "x": torch.zeros((count, n), device=dev, dtype=torch.float64)}
    if with_basis:
        out["basis"] = torch.zeros((count, m), dtype=torch.int64, device=dev)
        out["stats"] = torch.zeros((count, 8), dtype=torch.int32, device=dev)
    gm.simplex_batch_device(count, c.data_ptr(), A.data_ptr(), b.data_ptr(), m, n, tol, out["status"].data_ptr(),
                            out["optF"].data_ptr(), out["x"].data_ptr(),
                            out["basis"].data_ptr() if with_basis else 0,
                            out["stats"].data_ptr() if with_basis else 0, stream.cuda_stream)
    return out


def _device_matches(c, A, b, expect_tier, oracle_slice):
    import torch
    gm.init(0)
    dev = torch.device("cuda", 0)
    tc, tA, tb = (torch.from_numpy(v).to(dev) for v in (c, A, b))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        out = _device_call(tc, tA, tb, s)
        tier = gm.last_timing()["tier"]
        bare = _device_call(tc, tA, tb, s, with_basis=False)
    s.synchronize()
    d = {k: v.cpu().numpy() for k, v in out.items()}
    h = gm.simplex_batch(c, A, b)
    assert tier == expect_tier == gm.last_timing()["tier"], (tier, expect_tier)
    for k in ("status", "optF", "x", "basis"):
        assert np.array_equal(d[k], h[k]), k
    assert np.array_equal(d["stats"], h["stats"])
    for k in ("status", "optF", "x"):  # NULL basis / stats: same answers
        assert np.array_equal(bare[k].cpu().numpy(), d[k]), k
    count = len(c)
    sl = slice(0, oracle_slice)
    o = oracle.simplex_batch(c[sl], A[sl], b[sl], threads=oracle.num_hw_threads())
    assert (d["status"][sl] == o["status"]).all() and (d["status"] == S.GM_OK).all()
    assert rel(d["optF"][sl], o["optF"]) <= RTOL and rel(d["x"][sl], o["x"]) <= RTOL
    worst = Worst(f"device entry point {count} LPs {A.shape[1]}x{A.shape[2]}")
    for k in range(count):
        worst.add(tier_label(tier), check_certificate(c[k], A[k], b[k], d["basis"][k], d["x"][k]))
    worst.report()


@pytest.mark.timeout(600)
def test_device_entry_point_on_the_bench_workload():
    import bench
    c, A, b = bench.make_batch(0)
    assert A.shape == (4096, 64, 128)
    _device_matches(c, A, b, 1, 256)


@pytest.mark.timeout(600)
@pytest.mark.parametrize("m,n,count,tier", [(80, 170, 600, 2), (120, 250, 600, 3), (150, 300, 8, 6)])
def test_device_entry_point_on_other_tiers(m, n, count, tier):
    c, A, b = feasible_bounded_lp(np.random.default_rng(m + count), m, n, count)
    _device_matches(c, A, b, tier, 48)


@pytest.mark.timeout(300)
def test_device_entry_point_is_ordered_on_the_callers_stream():
    """The inputs are zero until a copy that a side stream enqueues behind a ~0.1 s spin; the engine call and the read
    of its outputs follow on the same stream. An engine that ran elsewhere would see zero rows."""
    import torch
    gm.init(0)
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(17)
    c, A, b = feasible_bounded_lp(rng, 64, 128, 512)
    src = [torch.from_numpy(v).to(dev) for v in (c, A, b)]
    dst = [torch.zeros_like(v) for v in src]
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
        for d_, s_ in zip(dst, src):
            d_.copy_(s_, non_blocking=True)
        out = _device_call(*dst, s)
        read = {k: v.clone() for k, v in out.items()}
    s.synchronize()
    h = gm.simplex_batch(c, A, b)
    assert (h["status"] == S.GM_OK).all()
    for k in ("status", "optF", "x", "basis"):
        assert np.array_equal(read[k].cpu().numpy(), h[k]), k


def test_device_entry_point_argument_codes():
    import torch
    gm.init(0)
    L = gm.capi.lib()
    dev = torch.device("cuda", 0)
    m, n = 4, 9
    c = torch.ones((1, n), dtype=torch.float64, device=dev)
    A = torch.ones((1, m, n), dtype=torch.float64, device=dev)
    b = torch.ones((1, m), dtype=torch.float64, device=dev)
    st = torch.full((1,), -7, dtype=torch.int32, device=dev)
    f = torch.zeros(1, dtype=torch.float64, device=dev)
    x = torch.zeros((1, n), dtype=torch.float64, device=dev)
    p = [t.data_ptr() for t in (c, A, b)]
    q = [t.data_ptr() for t in (st, f, x)]
    assert L.gm_simplex_batch_device(0, *p, m, n, 0.0, *q, None, None, None) == S.GM_OK
    torch.cuda.synchronize()
    assert int(st[0]) == -7  # nothing was written
    assert L.gm_simplex_batch_device(-1, *p, m, n, 0.0, *q, None, None, None) == S.GM_ERR_BAD_SHAPE
    for i in range(3):
        pp = list(p)
        pp[i] = None
        assert L.gm_simplex_batch_device(1, *pp, m, n, 0.0, *q, None, None, None) == S.GM_ERR_BAD_ARGUMENT
        qq = list(q)
        qq[i] = None
        assert L.gm_simplex_batch_device(1, *p, m, n, 0.0, *qq, None, None, None) == S.GM_ERR_BAD_ARGUMENT
    assert L.gm_simplex_batch_device(1, *p, 0, n, 0.0, *q, None, None, None) == S.GM_ERR_BAD_SHAPE


# ---- (f) early exits inside mixed batches ------------------------------------------------------------------------

MIXED = ([(70, t, 0) for t in (2, 3, 4, 5)] + [(130, t, 0) for t in (3, 4, 5)] +   # 130 x 270 does not fit tier 2
         [(m, 6, G) for m in (70, 130) for G in (1, 3)])


@pytest.mark.timeout(600)
@pytest.mark.parametrize("m,tier,G", MIXED, ids=[f"m{m}-tier{t}{f'-G{G}' if G else ''}" for m, t, G in MIXED])
def test_early_exits_inside_mixed_batches(m, tier, G):
    """Healthy LPs interleaved with LPs that exit before the main loop. With fewer LPs than CTAs / groups and with
    more, so that a CTA or group takes a healthy LP right after an early exit. Healthy LPs must be bitwise the
    answers of a batch without the early exits."""
    n = 2 * m + 10
    for count in (14, 400):
        c, A, b, kinds = mixed_batch(m, n, count, 1000 * m + count)
        g = solve(tier, G, c, A, b)
        grid = gm.last_timing()["grid"]
        units = grid // G if tier == 6 else grid  # groups of G CTAs, or persistent CTAs
        if tier == 6:
            assert (units < count) == (count == 400), (units, count)
        o = oracle_mixed(m, n, count, 1000 * m + count)
        assert (g["status"] == o["status"]).all(), [(k, kinds[k], g["status"][k], o["status"][k])
                                                    for k in np.nonzero(g["status"] != o["status"])[0]]
        for k, kind in enumerate(kinds):
            if kind in EXIT_STATUS:
                assert g["status"][k] == EXIT_STATUS[kind], (kind, g["status"][k])
        ok = np.array([k is None for k in kinds])
        assert (g["status"][ok] == S.GM_OK).all()
        assert rel(g["optF"][ok], o["optF"][ok]) <= RTOL and rel(g["x"][ok], o["x"][ok]) <= RTOL
        alone = solve(tier, G, c[ok], A[ok], b[ok])
        for key in ("status", "optF", "x", "basis", "pivots"):
            assert np.array_equal(alone[key], g[key][ok]), key
        print(f"m={m} {tier_label(tier, G)} count={count} on {units} CTAs / groups: statuses "
              f"{dict(zip(*np.unique(g['status'], return_counts=True)))} equal to the oracle's")


# ---- (h) reproducibility of tiers 5 and 6 --------------------------------------------------------------------------

@pytest.mark.timeout(300)
@pytest.mark.parametrize("tier,G", [(5, 0), (6, 3), (6, 37)], ids=["tier5", "tier6-G3", "tier6-G37"])
def test_tiers_5_and_6_are_bitwise_reproducible(tier, G):
    c, A, b = batch(120, 250, 64, 4242)
    runs = [solve(tier, G, c, A, b) for _ in range(3)]
    assert (runs[0]["status"] == S.GM_OK).all()
    for r in runs[1:]:
        for key in ("status", "optF", "x", "basis", "pivots"):
            assert np.array_equal(r[key], runs[0][key]), key
