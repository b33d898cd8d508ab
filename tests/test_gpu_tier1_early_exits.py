"""The register-resident tier (tier 1) on batches that mix healthy LPs with LPs that leave early (a zero
row, a zero column, Phase-I infeasible, unbounded, rank-deficient) and with LPs whose initial basis (the last m
columns) is exactly singular, at the elimination step chosen by the test.

Tier 1 reads each LP's A once, into shared memory, and runs the input checks there; its Gauss-Jordan inversion works
on registers. Statuses are compared with the CPU oracle, x and the objective at 1e-9 relative, and the answers of the
device-buffer entry point, the pageable host-buffer entry point and the pinned (streamed) host-buffer entry point must
be bitwise equal. The same batches run on the CPU through the emulated kernel (tests/emu), against the oracle."""
from functools import lru_cache

import numpy as np
import pytest

import emu_harness as E
import gomilp_b200 as gm
import oracle
from gomilp_b200 import status as S
from problems import feasible_bounded_lp

RTOL = 1e-9
KINDS = ("zero_row_b", "zero_row", "zero_col_neg", "zero_col", "phase1_infeasible", "unbounded", "dup_row",
         "singular_basis_first", "singular_basis_mid", "singular_basis_last")
# the statuses of the input checks (simplex.go:385-439), each with its first-index rule
EXIT_STATUS = {"zero_row_b": S.GM_ERR_INFEASIBLE, "zero_row": S.GM_ERR_ZERO_ROW, "zero_col_neg": S.GM_ERR_UNBOUNDED,
               "zero_col": S.GM_ERR_ZERO_COLUMN}


def rel(a, b) -> float:
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)))) if a.size else 0.0


def singular_last_block(rng, A, p1, p2):
    """Makes the block of the last m columns (basis position p = column n-1-p) exactly singular at elimination step p2:
    row r of the block is zero except at positions p1 < p2, and those two columns are 2 e_r and 4 e_r. No earlier
    step can pick row r or touch either column, step p1 pivots on row r, and at step p2 every candidate is 0."""
    m, n = A.shape
    r = int(rng.integers(m))
    A[r, n - m:] = 0.0
    A[:, n - 1 - p1] = 0.0
    A[:, n - 1 - p2] = 0.0
    A[r, n - 1 - p1], A[r, n - 1 - p2] = 2.0, 4.0


def early_exit_lp(rng, m, n, kind):
    c, A, b = feasible_bounded_lp(rng, m, n)
    i, j = int(rng.integers(m)), int(rng.integers(n))
    x0 = rng.random(n) * (rng.random(n) < 0.5)
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
        b = A @ x0
    elif kind == "dup_row":
        A[(i + 1) % m] = A[i]
        b = A @ x0
    elif kind.startswith("singular_basis"):
        # first: steps 0 and 1 (one register slot); mid: slots 2 and 9 (lane 1 of the quad); last: the last step
        p1, p2 = {"singular_basis_first": (0, 1), "singular_basis_mid": (9, min(37, m - 2)),
                  "singular_basis_last": (m // 2, m - 1)}[kind]
        singular_last_block(rng, A, p1, p2)
        b = A @ x0
        c = A.T @ rng.standard_normal(m) + rng.random(n)  # dual feasible again: bounded
    else:
        raise ValueError(kind)
    return c, A, b


@lru_cache(maxsize=None)
def mixed_batch(m, n, count, seed):
    """Even slots healthy LPs, odd slots the kinds above in turn. Returns c, A, b, kinds (None = healthy)."""
    rng = np.random.default_rng(seed)
    cs, As, bs, kinds = [], [], [], []
    for k in range(count):
        kind = None if k % 2 == 0 else KINDS[(k // 2) % len(KINDS)]
        c, A, b = feasible_bounded_lp(rng, m, n) if kind is None else early_exit_lp(rng, m, n, kind)
        cs.append(c), As.append(A), bs.append(b), kinds.append(kind)
    return np.array(cs), np.array(As), np.array(bs), tuple(kinds)


def device_call(c, A, b):
    import torch
    count, m, n = A.shape
    dev = torch.device("cuda", 0)
    tc, tA, tb = (torch.from_numpy(v).to(dev) for v in (c, A, b))
    out = {"status": torch.zeros(count, dtype=torch.int32, device=dev),
           "optF": torch.zeros(count, dtype=torch.float64, device=dev),
           "x": torch.zeros((count, n), dtype=torch.float64, device=dev),
           "basis": torch.zeros((count, m), dtype=torch.int64, device=dev),
           "stats": torch.zeros((count, 8), dtype=torch.int32, device=dev)}
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    gm.simplex_batch_device(count, tc.data_ptr(), tA.data_ptr(), tb.data_ptr(), m, n, 0.0, out["status"].data_ptr(),
                            out["optF"].data_ptr(), out["x"].data_ptr(), out["basis"].data_ptr(),
                            out["stats"].data_ptr(), s.cuda_stream)
    tier = gm.last_timing()["tier"]
    s.synchronize()
    return {k: v.cpu().numpy() for k, v in out.items()}, tier


def host_call(c, A, b, pinned):
    """gm_simplex_batch from pageable numpy buffers, or from pinned ones (a batch this size then streams)."""
    import ctypes as C
    import torch
    count, m, n = A.shape
    if pinned:
        keep = [torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for v in (c, A, b)]
        c, A, b = (t.numpy() for t in keep)
    out = {"status": np.zeros(count, np.int32), "optF": np.zeros(count), "x": np.zeros((count, n)),
           "basis": np.zeros((count, m), np.int64), "stats": np.zeros((count, 8), np.int32)}

    def p(a):
        return a.ctypes.data_as(C.c_void_p)

    rc = gm.capi.lib().gm_simplex_batch(count, p(c), p(A), p(b), m, n, 0.0, p(out["status"]), p(out["optF"]),
                                        p(out["x"]), p(out["basis"]), p(out["stats"]))
    assert rc == S.GM_OK, rc
    return out, gm.last_timing()["tier"]


def test_tier1_mixed_batches_emulated():
    for m, n, count in ((64, 128, 24), (33, 90, 20)):
        c, A, b, kinds = mixed_batch(m, n, count, 7000 + m + count)
        g = E.simplex_batch(c, A, b, reg=True)
        o = oracle.simplex_batch(c, A, b)
        assert (g["status"] == o["status"]).all(), [(k, kinds[k], g["status"][k], o["status"][k]) for k in
                                                    np.nonzero(g["status"] != o["status"])[0]]
        for k, kind in enumerate(kinds):
            if kind in EXIT_STATUS:
                assert g["status"][k] == EXIT_STATUS[kind], (k, kind, g["status"][k])
        ok = g["status"] == S.GM_OK
        assert all(ok[k] for k, kind in enumerate(kinds) if kind is None or kind.startswith("singular_basis"))
        assert rel(g["optF"][ok], o["optF"][ok]) <= RTOL and rel(g["x"][ok], o["x"][ok]) <= RTOL
        sing = np.array([kind is not None and kind.startswith("singular_basis") for kind in kinds])
        assert (g["stats"][sing, 5] & 1).all(), g["stats"][sing, 5]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("m,n,count", [(64, 128, 2400), (48, 110, 14), (33, 90, 300)],
                         ids=["64x128-2400", "48x110-14", "33x90-300"])
def test_tier1_mixed_batches_against_the_oracle_on_every_entry_point(m, n, count):
    gm.init(0)
    c, A, b, kinds = mixed_batch(m, n, count, 7000 + m + count)
    d, tier = device_call(c, A, b)
    assert tier == 1
    o = oracle.simplex_batch(c, A, b, threads=oracle.num_hw_threads())
    bad = np.nonzero(d["status"] != o["status"])[0]
    assert bad.size == 0, [(k, kinds[k], d["status"][k], o["status"][k]) for k in bad[:10]]
    for k, kind in enumerate(kinds):
        if kind in EXIT_STATUS:
            assert d["status"][k] == EXIT_STATUS[kind], (k, kind, d["status"][k])
    ok = d["status"] == S.GM_OK
    assert all(ok[k] for k, kind in enumerate(kinds) if kind is None or kind.startswith("singular_basis"))
    assert rel(d["optF"][ok], o["optF"][ok]) <= RTOL and rel(d["x"][ok], o["x"][ok]) <= RTOL
    sing = np.array([kind is not None and kind.startswith("singular_basis") for kind in kinds])
    # an exactly singular last block is not accepted: the column scan chooses the starting basis
    assert (d["stats"][sing, 5] & 1).all(), d["stats"][sing, 5]
    for pinned in (False, True):
        h, htier = host_call(c, A, b, pinned)
        assert htier == 1
        for key in ("status", "optF", "x", "basis", "stats"):
            assert np.array_equal(h[key], d[key], equal_nan=h[key].dtype.kind == "f"), (key, pinned)
    print(f"{m}x{n} count={count}: statuses {dict(zip(*np.unique(d['status'], return_counts=True)))} equal to the "
          f"oracle's; device, host and pinned host entry points bitwise equal")
