#!/usr/bin/env python
"""bench.py — LP relaxations solved per second on BASELINE.json configs[1]:
a batch of 4096 independent random dense LP relaxations, m=64, n=128, float64, per GPU (weak scaling).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N>1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

One "step" = one pass of the hot path (gm_simplex_batch_device: the simplex wave kernel) over one batch.
`value` is measured with the inputs resident in HBM; `e2e` goes through the host-buffer C-ABI entry point
(gm_simplex_batch) from pinned host memory, copies inside the timed region. `cpu_baseline` / `--impl
reference` time the CPU oracle (oracle/: C++ restatement of the reference's Gonum lp.Simplex — the
reference is Go and there is no Go toolchain in the image, so kind = "port") on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

M, N, BATCH = 64, 128, 4096
SEED = 1234
METRIC = "lp_relaxations_per_sec"
UNIT = "LP/s"
WORKLOAD = "C2: 4096 independent random dense LP relaxations m=64 n=128 f64 per GPU (feasible+bounded generator, seed 1234+rank)"


def hbm_tier_extra(gm):
    """The HBM-resident pivot path on BASELINE config 4's real shape, outside the timed region: (a) ONE dense LP
    m=1024 n=2048 (seed 42) solved to optimality by the cooperative tier with every SM on it; (b) a batch of 16 such
    LPs (seeds 42..57, working set 16 x 25 MB > L2) solved to optimality, groups of 9 CTAs per LP - the honest
    HBM-bound number. Everything reported is measured in this run."""
    try:
        from problems import feasible_bounded_lp
        m, n = 1024, 2048
        lps = [feasible_bounded_lp(np.random.default_rng(42 + k), m, n) for k in range(16)]
        c = np.stack([l[0] for l in lps]); A = np.stack([l[1] for l in lps]); b = np.stack([l[2] for l in lps])
        gm.simplex_batch(c[:1], A[:1], b[:1], want_basis=False)  # warm-up (loads the kernel)
        g1 = gm.simplex_batch(c[:1], A[:1], b[:1], want_basis=False)
        t1 = gm.last_timing()
        g16 = gm.simplex_batch(c, A, b, want_basis=False)
        t16 = gm.last_timing()
        p1, p16 = int(g1["pivots"].sum()), int(g16["pivots"].sum())
        bpp = bytes_per_pivot(m, n)
        peak = load_peaks().get("hbm_gbs", 6650.0)
        return {"single_lp": {"workload": "C4: one dense LP m=1024 n=2048 seed 42, solved to optimality",
                              "status_ok": bool((g1["status"] == 0).all()), "tier": t1["tier"], "grid": t1["grid"],
                              "pivots": p1, "kernel_ms": t1["kernel_ms"], "us_per_pivot": 1e3 * t1["kernel_ms"] / max(1, p1),
                              "algorithmic_GBps": p1 * bpp / (t1["kernel_ms"] * 1e-3) / 1e9,
                              "note": "working set 25 MB: L2 resident, so this is not an HBM figure"},
                "batch16": {"workload": "16 dense LPs m=1024 n=2048 seeds 42..57, solved to optimality (working set > L2)",
                            "status_ok": bool((g16["status"] == 0).all()), "tier": t16["tier"], "grid": t16["grid"],
                            "ctas_per_lp": t16["grid"] // 16, "pivots": p16, "kernel_ms": t16["kernel_ms"],
                            "bytes_per_pivot": bpp, "algorithmic_GBps": p16 * bpp / (t16["kernel_ms"] * 1e-3) / 1e9,
                            "frac_of_measured_hbm_peak": p16 * bpp / (t16["kernel_ms"] * 1e-3) / 1e9 / peak,
                            "note": "the fused update+FTRAN pass moves 2 m^2 + m(n-m) words per pivot, 0.75 of the "
                                    "3 m^2 + m(n-m) SURVEY 8(d) counts; inversions are inside the time"}}
    except Exception as e:
        gm.set_options()
        return {"error": repr(e)}


def load_peaks() -> dict:
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def bytes_per_pivot(m: int, n: int) -> int:
    """SURVEY.md §8(d): FTRAN reads B^-1 (m^2), the update reads+writes it (2 m^2), pricing reads A_N (m(n-m))."""
    return 8 * (3 * m * m + m * (n - m))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([s.strip() for s in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_batch(rank: int, count: int = BATCH):
    from problems import feasible_bounded_lp
    rng = np.random.default_rng(SEED + rank)
    return feasible_bounded_lp(rng, M, N, count)


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each output array of the last timed step as out_dir/<name>.npy in float64 (the integer outputs are
    small indices and counters, exact in float64), so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def cpu_baseline(count: int, threads: int):
    """The oracle timed on `count` LPs of the same workload with `threads` host threads."""
    import oracle
    c, A, b = make_batch(0, count)
    oracle.simplex_batch(c[:threads], A[:threads], b[:threads], threads=threads)  # warm the library
    t0 = time.perf_counter()
    o = oracle.simplex_batch(c, A, b, threads=threads)
    dt = time.perf_counter() - t0
    assert (o["status"] == 0).all()
    return count / dt, dt, int(o["pivots"].sum())


def bnb_extra(gm):
    """Second half of BASELINE.json's metric, outside the timed region: B&B nodes/s through gm_milp_solve on 1 GPU.
    (a) a small 0-1 knapsack (tier 1 waves) with the decisions replayed on the host and with the device-side scan;
    (b) BASELINE config 3's real shape, knapsack n=500 m=200 (700 x 1200 + depth), node-budgeted."""
    from problems import knapsack
    out = {}
    try:
        p = knapsack(np.random.default_rng(7), 30, 5)
        for warm_up_mode in (1, 1 | 4, 1 | 8):  # loads every kernel before anything is timed
            gm.milp_solve(p["c"], None, None, p["G"], p["h"], p["integrality"], mode=warm_up_mode, heuristic=1,
                          node_limit=256, keep_log=False)

        def best_of(prob, mode, limit, reps=3):
            best = None
            for _ in range(reps):
                t0 = time.perf_counter()
                res = gm.milp_solve(prob["c"], None, None, prob["G"], prob["h"], prob["integrality"], mode=mode,
                                    heuristic=1, node_limit=limit, keep_log=False)
                el = time.perf_counter() - t0
                if best is None or el < best[1]:
                    best = (res, el)
            return best

        def row(res, dt):
            return {"nodes_per_sec": res.nodes / dt, "nodes": res.nodes, "waves": res.waves, "pivots": res.pivots,
                    "wall_s": dt, "device_ms": res.device_ms, "status": res.status}

        out["small"] = {"workload": "0-1 knapsack n=30 m=5 (35x65 + depth), FIXED most-infeasible, node budget 8192, "
                                    "children solved cold like the reference, best of 3",
                        "host_replay": row(*best_of(p, 1, 8192)), "device_scan": row(*best_of(p, 1 | 8, 8192)),
                        "warm_start_host_replay": row(*best_of(p, 1 | 4, 8192))}
        p3 = knapsack(np.random.default_rng(7), 500, 200)
        r3, dt3 = best_of(p3, 1 | 8, 7, reps=1)
        out["c3"] = {"workload": "C3: 0-1 knapsack n=500 m=200 seed 7 (700x1200 + depth), FIXED most-infeasible, first 7 "
                                 "nodes (3 waves), device-side scan, cold children, reference rule set only (deeper "
                                 "nodes of this instance are degenerate enough that the reference's own arithmetic "
                                 "aborts, tests/golden/c3_knapsack.npz; bnb_sharded.c3 runs deeper with GM_BNB_ROBUST)",
                     **row(r3, dt3), "lp_status": r3.lp_status}
        from problems import c5_general_integer
        p5 = c5_general_integer(200)
        out["c5_n200"] = {"workload": "C5: general-integer MILP n=200 (300x500 + depth), FIXED most-infeasible, node budget "
                                      "511, device-side scan, cold children", **row(*best_of(p5, 1 | 8, 511, reps=2))}
        p51 = c5_general_integer(100)
        gm.milp_solve(p51["c"], None, None, p51["G"], p51["h"], p51["integrality"], mode=1 | 4 | 8, heuristic=1,
                      node_limit=512, keep_log=False)
        out["c5_n100"] = {"workload": "C5: general-integer MILP n=100 (150x250 + depth), FIXED most-infeasible, node budget "
                                      "16383, device-side scan, best of 2",
                          "cold_children": row(*best_of(p51, 1 | 8, 16383, reps=2)),
                          "warm_started_children": row(*best_of(p51, 1 | 4 | 8, 16383, reps=2)),
                          "note": "warm start (the north star's 'children warm-start from the parent basis'): every node's "
                                  "final basis and inverse stay in HBM, a child starts from [B 0; g 1]^-1; same optima, not "
                                  "a pivot-for-pivot replay of the reference's cold solves"}
    except Exception as e:  # never let the extra break the contract line
        out["error"] = repr(e)
    return out


def bnb_sharded_extra(gm, dist, dev, rank, world):
    """B&B frontier sharded over the ranks (gm_comm_init + gm_milp_solve_device): every rank calls with the same
    arguments, rank r solves the r-th FIFO block of every wave, one ncclAllGather of 32 B per node per wave."""
    import torch
    from problems import knapsack
    try:
        if world > 1:
            uid = torch.zeros(128, dtype=torch.uint8, device=dev)
            if rank == 0:
                uid = torch.frombuffer(bytearray(gm.capi.comm_unique_id()), dtype=torch.uint8).to(dev)
            dist.broadcast(uid, 0)
            gm.capi.comm_init(rank, world, bytes(uid.cpu().numpy().tobytes()))
        from problems import c5_general_integer

        def timed(prob, mode, limit, reps):
            best = None
            for rep in range(reps + 1):   # the first repetition is a warm-up (kernels, NCCL)
                if dist is not None:
                    dist.barrier()
                t0 = time.perf_counter()
                r = gm.milp_solve(prob["c"], None, None, prob["G"], prob["h"], prob["integrality"], mode=mode,
                                  heuristic=1, node_limit=limit, keep_log=False)
                dt = time.perf_counter() - t0
                if rep > 0 and (best is None or dt < best[1]):
                    best = (r, dt)
            r, dt = best
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            if dist is not None:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return {"nodes": r.nodes, "waves": r.waves, "pivots": r.pivots, "status": r.status, "lp_status": r.lp_status,
                    "wall_s_max_over_ranks": float(t[0]), "nodes_per_sec": r.nodes / float(t[0]), "device_ms": r.device_ms}

        out = {"gpus": world,
               "collective": "ncclAllGather of 32-byte node records, once per wave" if world > 1 else "none",
               "c5_n100": {"workload": "C5 general-integer MILP n=100 (150x250 + depth, bounds as rows), FIXED "
                                       "most-infeasible, node budget 65535, device-side scan, FIFO blocks per rank, cold "
                                       "children, best of 2 after a warm-up run",
                           **timed(c5_general_integer(100), 1 | 8, 65535, 2)},
               "c3": {"workload": "C3: 0-1 knapsack n=500 m=200 seed 7 (700x1200 + depth), FIXED most-infeasible, node "
                                  "budget 127, device-side scan, FIFO blocks per rank, cold children, GM_BNB_ROBUST (the "
                                  "reference's own rule set aborts on this instance's children beyond depth 2), best of 1 "
                                  "after a warm-up run",
                      **timed(knapsack(np.random.default_rng(7), 500, 200), 1 | 8 | 16, 127, 1)}}
        if world > 1:
            gm.capi.comm_destroy()
        return out
    except Exception as e:
        return {"error": repr(e)}


def base_config() -> dict:
    """The workload description both arms print (identical, so that the driver sees the same config)."""
    return {"workload": WORKLOAD, "m": M, "n": N, "batch_per_gpu": BATCH, "tol": 0.0,
            "l2": "inputs (275 MB per GPU) exceed the 126 MB L2; no explicit flush",
            "sharding": "independent LPs, no data-path collective"}


def run_reference(args, rank: int, world: int):
    """The reference's CPU path (oracle/: C++ restatement of Gonum's lp.Simplex, the Go toolchain being absent) on the
    box's host cores, all of them, on the SAME 4096-LP batch. A step is the whole batch when the run then still ends
    within a few minutes at the rate measured during warm-up, else the largest prefix of the batch that does."""
    if rank != 0:
        return
    import oracle
    cores = os.cpu_count() or 1
    c, A, b = make_batch(0, BATCH)
    nw = min(BATCH, 8 * cores)
    rate = None
    for _ in range(max(1, args.warmup)):
        t0 = time.perf_counter()
        oracle.simplex_batch(c[:nw], A[:nw], b[:nw], threads=cores)
        rate = nw / (time.perf_counter() - t0)
    per_step = int(min(BATCH, max(8 * cores, rate * 200.0 / max(1, args.steps))))
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o = oracle.simplex_batch(c[:per_step], A[:per_step], b[:per_step], threads=cores)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: o[k] for k in ("status", "optF", "x", "basis")})
    value = per_step * args.steps / dt
    sample = (f"the first {per_step} of the batch's {BATCH} LPs per step, {cores} threads, one LP per thread"
              if per_step < BATCH else f"the whole {BATCH}-LP batch per step, {cores} threads, one LP per thread")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps * (BATCH / per_step),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def run_ours(args, rank: int, world: int, local_rank: int):
    import torch
    import gomilp_b200 as gm
    if not torch.cuda.is_available() or gm.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    gm.init(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        dist.init_process_group("nccl", device_id=dev)

    c, A, b = make_batch(rank)
    # pinned host copies (e2e) and device-resident copies (value)
    hc = torch.from_numpy(c).pin_memory()
    hA = torch.from_numpy(A).pin_memory()
    hb = torch.from_numpy(b).pin_memory()
    dc, dA, db = hc.to(dev), hA.to(dev), hb.to(dev)
    d_status = torch.zeros(BATCH, dtype=torch.int32, device=dev)
    d_optF = torch.zeros(BATCH, dtype=torch.float64, device=dev)
    d_x = torch.zeros(BATCH, N, dtype=torch.float64, device=dev)
    d_basis = torch.zeros(BATCH, M, dtype=torch.int64, device=dev)
    d_stats = torch.zeros(BATCH, 8, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)

    def step():
        gm.simplex_batch_device(BATCH, dc.data_ptr(), dA.data_ptr(), db.data_ptr(), M, N, 0.0, d_status.data_ptr(),
                                d_optF.data_ptr(), d_x.data_ptr(), d_basis.data_ptr(), d_stats.data_ptr(),
                                stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    with torch.cuda.stream(stream):
        ev[0].record(stream)
        for k in range(args.steps):
            step()
            ev[k + 1].record(stream)
    stream.synchronize()
    barrier()
    total_ms = ev[0].elapsed_time(ev[-1])
    kernel_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    tm = gm.last_timing()
    status = d_status.cpu().numpy()
    stats = d_stats.cpu().numpy()
    pivots = int(stats[:, 0].sum() + stats[:, 1].sum())
    inversions = int(stats[:, 3].sum())
    assert (status == 0).all(), "bench workload must solve to optimality"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"status": status, "optF": d_optF.cpu().numpy(), "x": d_x.cpu().numpy(),
                                         "basis": d_basis.cpu().numpy(), "stats": stats})

    # ---- e2e: host buffers through the C ABI, copies inside the timed region --------------------
    # results land in pinned host memory too (a device->host copy into pageable memory is staged and ~4x slower)
    hs = torch.zeros(BATCH, dtype=torch.int32).pin_memory().numpy()
    hF = torch.zeros(BATCH, dtype=torch.float64).pin_memory().numpy()
    hx = torch.zeros(BATCH, N, dtype=torch.float64).pin_memory().numpy()
    hB = torch.zeros(BATCH, M, dtype=torch.int64).pin_memory().numpy()
    hS = torch.zeros(BATCH, 8, dtype=torch.int32).pin_memory().numpy()
    cn, An, bn = hc.numpy(), hA.numpy(), hb.numpy()
    import ctypes as C
    L = gm.capi.lib()

    def p(a):
        return a.ctypes.data_as(C.c_void_p)

    if args.no_streamed:
        gm.set_options(no_streamed_batch=True)

    def e2e_step():
        rc = L.gm_simplex_batch(BATCH, p(cn), p(An), p(bn), M, N, 0.0, p(hs), p(hF), p(hx), p(hB), p(hS))
        assert rc == 0, rc

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    e2e_tm = gm.last_timing()
    gm.set_options()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    assert np.array_equal(hs, status) and np.allclose(hF, d_optF.cpu().numpy(), rtol=0, atol=0)

    t = torch.tensor([total_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pv = torch.tensor([pivots], dtype=torch.float64, device=dev)
        dist.all_reduce(pv)
        pivots_all = int(pv.item())
    else:
        pivots_all = pivots
    total_ms, e2e_ms = float(t[0]), float(t[1])
    # extras, outside the timed region. The sharded B&B is collective: every rank takes part.
    bnb_sh = bnb_sharded_extra(gm, dist, dev, rank, world) if not args.quick else {"skipped": "--quick"}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    smem_peak = gm.capi.microbench_smem_gbs()
    bnb = bnb_extra(gm) if not args.quick else {"skipped": "--quick"}
    hbm_tier = hbm_tier_extra(gm) if not args.quick else {"skipped": "--quick"}

    value = world * BATCH * args.steps / (total_ms * 1e-3)
    e2e_value = world * BATCH * args.steps / (e2e_ms * 1e-3)
    peaks = load_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    launch_ms = float(np.mean(kernel_ms))
    alg_bytes = pivots * bytes_per_pivot(M, N)  # this rank's launch
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    cores = os.cpu_count() or 1
    n_cpu = BATCH  # the whole batch: ~6 s of wall clock on 16 cores (~100 core-seconds)
    cpu_v, cpu_dt, _ = cpu_baseline(n_cpu, cores)
    h2d = BATCH * (M * N + M + N) * 8
    d2h = BATCH * (N + 1) * 8 + BATCH * 4 + BATCH * M * 8 + BATCH * 8 * 4
    traffic, traffic_src = None, "null: no ncu capture of this round found under profiles/"
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
            tr = json.load(f)["simplex_wave_reg"]
        traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
        traffic_src = ("NOT measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of one launch of this "
                       "workload from the committed ncu --set full capture " + tr["source"])
    except Exception:
        pass
    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(),
        "detail": {"tier": tm["tier"], "grid": tm["grid"], "block": tm["block"], "smem_bytes_per_cta": tm["smem_bytes"],
                   "pivots_per_lp": pivots / BATCH, "basis_inversions_per_lp": inversions / BATCH},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps,
                "breakdown_last_step_ms": {"h2d": e2e_tm["h2d_ms"], "kernel": e2e_tm["kernel_ms"], "d2h": e2e_tm["d2h_ms"]},
                "api": "gm_simplex_batch (C ABI, pinned host buffers)",
                "launches_last_step": e2e_tm["launches"],
                "path": "one launch per slice" if args.no_streamed else "one launch, CTAs gated on the copy stream's "
                        "arrival counter (the batch crosses PCIe while the first LPs are being solved)"},
        "gpu_launches": args.steps,
        # Tier 1 keeps B^-1 in registers and W in shared memory: the per-pivot bytes never reach HBM (the batch is
        # read from HBM once per launch), so the roof that bounds this kernel is the SM's shared-memory / issue
        # bandwidth. `achieved` = SURVEY 8(d)'s algorithmic bytes per pivot x pivots per launch / launch time,
        # `peak` = the shared-memory bandwidth MEASURED in this run by gm_microbench_smem_gbs.
        "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s",
                     "frac": achieved / smem_peak if smem_peak else None, "traffic": traffic,
                     "kernel": "simplex_wave_reg", "launch_ms": launch_ms,
                     "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_pivot": bytes_per_pivot(M, N),
                     "pivots_per_launch": pivots,
                     "peak_source": "measured in this run: all SMs streaming conflict-free 16-byte shared-memory loads "
                                    "(gm_microbench_smem_gbs); theoretical 148 SMs x 128 B/clk x 1.965 GHz = 37.2 TB/s",
                     "hbm": {"one_off_bytes_per_launch": BATCH * (M * N + M + N + N + 1 + M) * 8,
                             "one_off_GBps": BATCH * (M * N + M + N + N + 1 + M) * 8 / (launch_ms * 1e-3) / 1e9,
                             "peak": hbm_peak, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks
                             else "fallback",
                             "note": "dram traffic of this kernel is the batch read once + results written once; "
                                     "ncu dram__bytes captures live under profiles/, not in this line"},
                     "traffic_source": traffic_src},
        "cpu_baseline": {"value": cpu_v, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"all {n_cpu} LPs of rank 0's batch, {cores} threads, {cpu_dt:.1f} s of wall clock"},
        "pivots_per_sec": pivots_all * args.steps / (total_ms * 1e-3),
        "bnb": bnb,
        "bnb_sharded": bnb_sh,
        "hbm_tier": hbm_tier,
        "clocks": clocks,
    }))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="skip the B&B / HBM-tier extras (profiling runs)")
    ap.add_argument("--no-streamed", action="store_true",
                    help="e2e through one launch per slice instead of one launch gated on arrival counters: required "
                         "under ncu, whose kernel replay serialises launches (a kernel that waits for a copy issued "
                         "after it would never see it)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the arrays the last step returned (rank 0's; with --impl "
                         "reference, those of the batch prefix it solves) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under it so that there is one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29533"),
               os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup",
               str(args.warmup), "--impl", args.impl] + (["--quick"] if args.quick else []) + \
              (["--no-streamed"] if args.no_streamed else []) + \
              (["--dump-outputs", os.path.abspath(args.dump_outputs)] if args.dump_outputs else [])
        sys.exit(subprocess.call(cmd))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
