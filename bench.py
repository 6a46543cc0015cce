#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 leapfrog engine (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch: the fused L=32-step leapfrog trajectory
(`step(Leapfrog(0.1), h, z, 32)`, src/integrator.jl:216-265) of 4096 chains x D=128 on a diagonal Gaussian
target with a Diag-Euclidean metric -- the configuration BASELINE.json's metric is quoted on.
Metric: leapfrog-steps*dims/s.  Weak scaling: every rank runs the same 4096-chain batch (chains shard
with no data-path collective, SURVEY 8e), value = all ranks' units / max-over-ranks device time.

--dump-outputs DIR writes the phase point the last timed step returned (rank 0; float64, 12.6 MB) as DIR/<name>.npy.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
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

N_CHAINS, DIM, L_STEPS, EPS = 4096, 128, 32, 0.1
METRIC_NAME = "leapfrog-steps*dims/sec"
WORKLOAD = "north-star headline: 4096 chains x D=128 diag-Gaussian (s log-spaced 0.1..10), DiagEuclidean Minv=s^2, Leapfrog(0.1), L=32 fused steps per launch"
SEED = 20260923


def config_dict(world):
    """the SAME keys and values in both arms (the driver compares the two `config` objects)"""
    return {"workload": WORKLOAD, "chains_per_gpu": N_CHAINS, "D": DIM, "L": L_STEPS, "eps": EPS,
            "parallelism": f"chains sharded x{world}, no data-path collective",
            "l2": "flushed between timed iterations (512 MiB read-sweep outside the event pair)"}


def synth(N, D, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    s = np.exp(np.linspace(np.log(0.1), np.log(10.0), D))
    m = np.zeros(D)
    th = rng.normal(size=(N, D))
    r = rng.normal(size=(N, D)) / s
    return m, s, s * s, th, r


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    try:
        with open(os.path.join(ROOT, "profiles", "r02", "k1_headline_dram.json")) as f:
            d = json.load(f)
        return int(d["dram_bytes_read"] + d["dram_bytes_write"])
    except Exception:
        return None


def save_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), np.ascontiguousarray(v, dtype=np.float64))


class Extra:
    """an extra measurement that fails is reported under "extras_failed" -- it must never cost the headline line"""
    errors = {}

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        return self

    def __exit__(self, et, ev, tb):
        if et is not None and issubclass(et, Exception):
            Extra.errors[self.name] = f"{et.__name__}: {ev}"[:300]
            return True
        return False


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        self.proc.wait()
        sm, reasons, mx = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
def cpu_baselines(m, s, Minv, th, r, full=True):
    """Timed CPU restatements of the same workload on this box's host cores (oracle/ = test+bench infra).
    numpy twin = op-for-op with the reference's temporaries, single thread like Julia's broadcast;
    C/OpenMP = fused good-CPU bound, all cores."""
    from oracle import oracle_c as oc
    from oracle import oracle_np as onp

    N, D = th.shape
    units = N * D * L_STEPS
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s), oc.Metric(oc.DIAG, Minv)
    z0 = oc.phasepoint(om, ome, th.T, r.T)
    out = oc.PhasePoint(D, N, with_lk_gradient=False)
    cores, best = best_threads(lambda nt: oc.leapfrog_omp(om, ome, EPS, z0, L_STEPS, n_threads=nt, out=out))
    res = {"omp": units / best, "cores": cores}
    if full:
        nm, nme = onp.Model(onp.DIAG_GAUSS, D, m, s), onp.Metric(onp.DIAG, Minv)
        y0 = onp.phasepoint(nm, nme, np.asfortranarray(th.T), np.asfortranarray(r.T))
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            onp.step(nm, nme, EPS, y0, L_STEPS)
            ts.append(time.perf_counter() - t0)
        res["numpy_1thread"] = units / float(np.median(ts))
    return res


def host_threads():
    """threads this process may actually use: min(affinity mask, cgroup cpu quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(p))))
    except Exception:
        pass
    return n


def best_threads(fn):
    """pick the OpenMP thread count (powers of two up to host_threads()) that runs `fn` fastest:
    'all the host threads it can use' without oversubscribing a quota-limited container."""
    cap = host_threads()
    cands = sorted({min(cap, 1 << k) for k in range(0, 9)} | {cap})
    best_t, best_n = None, 1
    for nt in cands:
        fn(nt)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            fn(nt)
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        if best_t is None or t < best_t:
            best_t, best_n = t, nt
    return best_n, best_t


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The Julia reference cannot
    run here (no julia binary, nothing to compile into oracle/_ref), so this arm times the oracle port
    with all host threads (fused C/OpenMP) and reports the single-thread op-for-op numpy twin beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, s, Minv, th, r = synth(N_CHAINS, DIM, SEED)
    from oracle import oracle_c as oc

    om, ome = oc.Model(oc.DIAG_GAUSS, DIM, m, s), oc.Metric(oc.DIAG, Minv)
    z0 = oc.phasepoint(om, ome, th.T, r.T)
    out = oc.PhasePoint(DIM, N_CHAINS, with_lk_gradient=False)
    units = N_CHAINS * DIM * L_STEPS
    cores, _ = best_threads(lambda nt: oc.leapfrog_omp(om, ome, EPS, z0, L_STEPS, n_threads=nt, out=out))
    for _ in range(args.warmup):
        oc.leapfrog_omp(om, ome, EPS, z0, L_STEPS, n_threads=cores, out=out)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oc.leapfrog_omp(om, ome, EPS, z0, L_STEPS, n_threads=cores, out=out)
    dt = time.perf_counter() - t0
    # the oracle's (D, N) column-major arrays, stored in the (N, D) layout of the GPU arm; this arm's model has no
    # normalising constant, so its lp_value differs from the GPU arm's by -D/2 log(2 pi) - sum(log s)
    if args.dump_outputs:
        save_outputs(args.dump_outputs, {"theta": out.theta.T, "r": out.r.T, "lp_value": out.lp_value,
                                         "lp_gradient": out.lp_gradient.T, "lk_value": out.lk_value})
    value = units * args.steps / dt
    extra = cpu_baselines(m, s, Minv, th, r, full=True)
    line = {
        "impl": "reference", "metric": METRIC_NAME, "value": value, "unit": "steps*dims/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(args.gpus),
        "cpu_baseline": {"value": value, "unit": "steps*dims/s", "cores": cores, "kind": "port",
                         "sample": "full workload per step (4096x128x32), fused C/OpenMP oracle port, all host threads; "
                                   "the Julia reference itself cannot run here (no julia binary)",
                         "numpy_twin_1thread": extra.get("numpy_1thread")},
        "e2e": {"value": value, "unit": "steps*dims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    args.emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    import ahmc_b200 as A

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    ctx = A.get_context(local, stream=stream.cuda_stream)
    hbm_peak, peak_src = peaks()

    m, s, Minv, th, r = synth(N_CHAINS, DIM, SEED + rank)
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s))
    lf = A.Leapfrog(EPS)
    K, W = args.steps, args.warmup
    units_per_step = N_CHAINS * DIM * L_STEPS

    with torch.cuda.stream(stream):
        z0 = A.phasepoint(h, torch.as_tensor(th, device=dev), torch.as_tensor(r, device=dev))
        flush = torch.zeros(512 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)  # 512 MiB > 126 MB L2

        def flush_l2():
            # READ 512 MiB: fills L2 with clean lines of another buffer (a write-flush would leave it full of
            # dirty lines whose write-back is then billed to the timed kernel)
            return flush.max()

        # prepared call: one foreign call per step, so the host stays ahead of the ~10 us kernel and the
        # CUDA-event pair brackets device execution only
        one_step = A.StepPlan(lf, h, z0, L_STEPS, flags=A.FLAG_ASYNC)

        for _ in range(max(W, 3)):
            flush_l2()
            one_step()
        stream.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local)
        sampler.start()
        try:
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
            l0 = ctx.launches
            for i in range(K):
                flush_l2()  # L2 flush between timed iterations (outside the event pair)
                ev[i][0].record(stream)
                zt = one_step()
                ev[i][1].record(stream)
            dumped = None
            if args.dump_outputs and rank == 0:  # copied on the stream before the untimed steps below overwrite them
                dumped = {"theta": zt.theta.clone(), "r": zt.r.clone(), "lp_value": zt.lp.value.clone(),
                          "lp_gradient": zt.lp.gradient.clone(), "lk_value": zt.lk.value.clone()}
            torch.cuda.synchronize()
            launches = ctx.launches - l0
            # keep the sampler alive for a moment of sustained load so clocks are seen under load
            t_end = time.time() + 0.4
            while time.time() < t_end:
                one_step()
            torch.cuda.synchronize()
        finally:
            clocks = sampler.stop()
        if dumped is not None:
            save_outputs(args.dump_outputs, {k: v.cpu().numpy() for k, v in dumped.items()})
        if world > 1:
            dist.barrier()
        step_ms = [a.elapsed_time(b) for a, b in ev]
        dev_ms = float(sum(step_ms))

        # ---- HBM-honest shape: 2^20 chains x D=128, ONE leapfrog step per launch, in place (3 GiB of state)
        honest = None
        if rank == 0 and not args.no_extras:
            with Extra("honest"):
                Nh = 1 << 20
                g = torch.Generator(device=dev).manual_seed(1)
                st = torch.as_tensor(s, device=dev)
                zh = A.phasepoint(h, torch.randn((Nh, DIM), generator=g, dtype=torch.float64, device=dev) * st,
                                  torch.randn((Nh, DIM), generator=g, dtype=torch.float64, device=dev) / st)
                import ctypes as C

                md, keep = h.metric._desc(DIM, Nh, zh.theta)
                zc = zh._c(False)
                call = lambda: ctx.check(ctx.lib.ahmc_leapfrog_f64(ctx.h, h.target.handle(ctx), C.byref(md), DIM, Nh, EPS, None, 1,
                                                                   0.0, C.byref(zc), C.byref(zc), None, None, A.FLAG_ASYNC))
                for _ in range(3):
                    call()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                reps = 10
                e0.record(stream)
                for _ in range(reps):
                    call()
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                bytes_launch = Nh * DIM * 48 + Nh * 16
                honest = {"workload": "2^20 chains x D=128, 1 step per launch, in place (3 GiB state >> L2)",
                          "ms_per_launch": ms, "achieved": bytes_launch / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
                          "frac": bytes_launch / ms / 1e6 / hbm_peak, "rate_steps_dims_per_s": Nh * DIM / ms * 1e3}
                # ---- same kernel, fused L=32 steps at 2^20 chains: the large-batch regime where launch overhead is
                # amortised and the register-resident trajectory is bound by its COMPULSORY HBM traffic
                callL = lambda: ctx.check(ctx.lib.ahmc_leapfrog_f64(ctx.h, h.target.handle(ctx), C.byref(md), DIM, Nh, EPS, None,
                                                                    L_STEPS, 0.0, C.byref(zc), C.byref(zc), None, None, A.FLAG_ASYNC))
                callL()
                e0.record(stream)
                for _ in range(5):
                    callL()
                e1.record(stream)
                torch.cuda.synchronize()
                msL = e0.elapsed_time(e1) / 5
                honest["fused_L32"] = {"workload": "2^20 chains x D=128, L=32 fused steps per launch, in place",
                                       "ms_per_launch": msL, "rate_steps_dims_per_s": Nh * DIM * L_STEPS / msL * 1e3,
                                       "achieved_compulsory": bytes_launch / msL / 1e6, "frac_compulsory": bytes_launch / msL / 1e6 / hbm_peak,
                                       "fp64_tflops": Nh * DIM * L_STEPS * 4 / msL / 1e9}
                del zh

        # ---- fixed vs marginal cost of the headline launch: the same fused L=32 launch at 4x the chains, same cold-L2 protocol.
        # (t_16384 - t_4096) / 3 is what 4096 more chains cost once the launch is under way; the rest is launch + cold start.
        batch = None
        if rank == 0 and not args.no_extras:
            with Extra("batch"):
                Nb = 4 * N_CHAINS
                mb_, sb_, Minvb, thb, rb = synth(Nb, DIM, SEED + 99)
                zb = A.phasepoint(h, torch.as_tensor(thb, device=dev), torch.as_tensor(rb, device=dev))
                planb = A.StepPlan(lf, h, zb, L_STEPS, flags=A.FLAG_ASYNC)
                for _ in range(3):
                    flush_l2()
                    planb()
                evb = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(10)]
                for a_, b_ in evb:
                    flush_l2()
                    a_.record(stream)
                    planb()
                    b_.record(stream)
                torch.cuda.synchronize()
                t4 = float(np.median([a_.elapsed_time(b_) for a_, b_ in evb])) * 1e3  # us
                t1 = float(np.median(step_ms)) * 1e3
                marg = (t4 - t1) / 3.0
                comp = N_CHAINS * DIM * 48 + N_CHAINS * 24
                batch = {"what": "median CUDA-event time of the fused L=32 launch at 4096 and at 16384 chains, L2 flushed before each",
                         "us_4096": t1, "us_16384": t4, "marginal_us_per_4096_chains": marg, "fixed_us": t1 - marg,
                         "marginal_compulsory_GBps": comp / marg / 1e3, "marginal_frac_of_hbm": comp / marg / 1e3 / hbm_peak}

        # ---- K2: fused static-HMC transition (refresh + 32 steps + MH) on the same batch
        k2 = None
        if rank == 0 and not args.no_extras:
            with Extra("k2"):
                kern = A.HMCKernel(A.Trajectory(A.EndPointTS, lf, A.FixedNSteps(L_STEPS)))
                prng = A.PhiloxRNG(7)
                NT = 100  # transitions per chain inside ONE launch (ahmc_hmc_sample_f64): no host work between transitions
                for _ in range(2):
                    A.sample_transitions(prng, h, kern, z0, NT, keep_draws=False)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record(stream)
                A.sample_transitions(prng, h, kern, z0, NT, keep_draws=False, flags=A.FLAG_ASYNC)
                e1.record(stream)
                torch.cuda.synchronize()
                ms_k2 = e0.elapsed_time(e1) / NT
                k2 = {"workload": "static HMC transitions (Philox refresh + 32 fused steps + MH), 4096x128, 100 transitions per chain in one launch",
                      "ms_per_transition": ms_k2, "rate_steps_dims_per_s": units_per_step / ms_k2 * 1e3}

        # ---- the GENERAL path on the same shape: per-step reference op sequence with energies and isfinite tests (what every
        # non-Gaussian user model runs), the funnel target, and NUTS on the C3 shape (persistent launch, 20 transitions)
        general = None
        if rank == 0 and not args.no_extras:
            with Extra("general"):
                general = {}
                B = 48.0 + 24.0 / DIM

                def timed(fn, reps):
                    for _ in range(3):
                        fn()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(reps):
                        fn()
                    e1.record(stream)
                    torch.cuda.synchronize()
                    return e0.elapsed_time(e1) / reps

                ex = A.StepPlan(lf, h, z0, L_STEPS, flags=A.FLAG_ASYNC | A.FLAG_EXACT_CHECKS)
                ms = timed(ex, 20)
                rate = units_per_step / ms * 1e3
                general["exact_path"] = {"workload": "headline shape, AHMC_FLAG_EXACT_CHECKS: per-step energies + isfinite, no linear shortcut",
                                         "ms_per_launch": ms, "rate_steps_dims_per_s": rate, "roofline_frac_contract": rate * B / 1e9 / hbm_peak,
                                         "roofline_frac_compulsory": (N_CHAINS * DIM * 48 + N_CHAINS * 24) / ms / 1e6 / hbm_peak}
                Df = 100
                hf = A.Hamiltonian(A.DiagEuclideanMetric(np.ones(Df)), A.Funnel(Df))
                gf = torch.Generator(device=dev).manual_seed(3)
                zf = A.phasepoint(hf, 0.5 * torch.randn((N_CHAINS, Df), generator=gf, dtype=torch.float64, device=dev),
                                  torch.randn((N_CHAINS, Df), generator=gf, dtype=torch.float64, device=dev))
                fp = A.StepPlan(A.Leapfrog(0.05), hf, zf, L_STEPS, flags=A.FLAG_ASYNC)
                ms = timed(fp, 20)
                rate = N_CHAINS * Df * L_STEPS / ms * 1e3
                Bf = 48.0 + 24.0 / Df
                general["funnel_trajectory"] = {"workload": "Neal's funnel D=100 (SURVEY 8c), 4096 chains, Diag metric, Leapfrog(0.05), L=32 fused",
                                                "ms_per_launch": ms, "rate_steps_dims_per_s": rate, "roofline_frac_contract": rate * Bf / 1e9 / hbm_peak,
                                                "roofline_frac_compulsory": (N_CHAINS * Df * 48 + N_CHAINS * 24) / ms / 1e6 / hbm_peak}
                kn = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.4), A.GeneralisedNoUTurn()))
                prn = A.PhiloxRNG(11)
                zs = A.phasepoint(h, torch.as_tensor(th * s, device=dev), torch.as_tensor(r, device=dev))  # theta ~ target
                TN = 20
                zl, _, stn = A.sample_transitions(prn, h, kn, zs, TN, keep_draws=False, flags=A.FLAG_ASYNC)
                torch.cuda.synchronize()
                reps_n = []
                for _ in range(3):  # three launches of 20 transitions each: median (a ~40-100 ms launch right after host work
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)  # is sensitive to clock ramp-up)
                    e0.record(stream)
                    zl, _, stn = A.sample_transitions(prn, h, kn, zl, TN, keep_draws=False, flags=A.FLAG_ASYNC)
                    e1.record(stream)
                    torch.cuda.synchronize()
                    reps_n.append((e0.elapsed_time(e1), int(stn["n_steps"].sum().item())))
                reps_n.sort(key=lambda t: t[0] / t[1])
                msn, nsteps = reps_n[1]
                rate = nsteps * DIM / msn * 1e3
                general["nuts_c3"] = {"workload": "C3: NUTS(MultinomialTS, GeneralisedNoUTurn) + DiagEuclidean, D=128 Gaussian, 4096 chains, eps=0.4, "
                                                  "20 transitions per chain in one persistent launch",
                                      "ms_per_transition": msn / TN, "ms_per_transition_all_reps": [t[0] / TN for t in reps_n],
                                      "mean_leapfrog_steps_per_transition": nsteps / TN / N_CHAINS,
                                      "rate_steps_dims_per_s": rate, "roofline_frac_contract": rate * B / 1e9 / hbm_peak}

                # C5's shape on this GPU: NUTS with DENSE operators (Dense metric = Sigma, dense-precision Gaussian, D = 256): the
                # block-cooperative form -- 8 chains share every D x D product (bulk-copied column chunks, fp64 MMA)
                D5, N5, T5 = 256, 8192, 5
                rng5 = np.random.Generator(np.random.PCG64(SEED + 5))
                Q5, _ = np.linalg.qr(rng5.normal(size=(D5, D5)))
                lam5 = np.exp(np.linspace(np.log(0.1), np.log(10.0), D5))
                Sig5, P5 = (Q5 * lam5) @ Q5.T, (Q5 / lam5) @ Q5.T
                h5 = A.Hamiltonian(A.DenseEuclideanMetric(Sig5), A.DenseGaussian(np.zeros(D5), P5))
                k5 = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.5), A.GeneralisedNoUTurn()))
                g5 = torch.Generator(device=dev).manual_seed(5)
                th5 = torch.randn((N5, D5), generator=g5, dtype=torch.float64, device=dev)
                z5 = A.phasepoint(h5, th5, torch.zeros_like(th5))
                p5 = A.PhiloxRNG(12)
                z5, _, st5 = A.sample_transitions(p5, h5, k5, z5, T5, keep_draws=False, flags=A.FLAG_ASYNC)
                torch.cuda.synchronize()
                reps5 = []
                for _ in range(3):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    z5, _, st5 = A.sample_transitions(p5, h5, k5, z5, T5, keep_draws=False, flags=A.FLAG_ASYNC)
                    e1.record(stream)
                    torch.cuda.synchronize()
                    reps5.append((e0.elapsed_time(e1), int(st5["n_steps"].sum().item())))
                reps5.sort(key=lambda t: t[0] / t[1])
                ms5, ns5 = reps5[1]
                rate5 = ns5 * D5 / ms5 * 1e3
                general["nuts_c5"] = {"workload": "C5 shape: NUTS + DenseEuclidean (M^-1 = Sigma) on a dense-precision Gaussian, D=256, 8192 chains, "
                                                  "eps=0.5, 5 transitions per chain in one persistent launch (median of 3 launches)",
                                      "ms_per_transition": ms5 / T5, "mean_leapfrog_steps_per_transition": ns5 / T5 / N5,
                                      "rate_steps_dims_per_s": rate5,
                                      "fp64_mma_tflops": rate5 * 4 * D5 / 1e12}  # two D x D products per leaf = 4 D flop per step x dim

        # ---- K4: correlated (dense-precision) Gaussian target, Diag metric, same batch: fp64 tensor-MMA trajectory
        k4 = None
        if rank == 0 and not args.no_extras:
            with Extra("k4"):
                rng4 = np.random.Generator(np.random.PCG64(SEED))
                Q, _ = np.linalg.qr(rng4.normal(size=(DIM, DIM)))
                lam = np.exp(np.linspace(np.log(0.1), np.log(10.0), DIM))
                hd = A.Hamiltonian(A.DiagEuclideanMetric(np.diag((Q * lam) @ Q.T).copy()), A.DenseGaussian(np.zeros(DIM), (Q / lam) @ Q.T))
                zd = A.phasepoint(hd, torch.as_tensor(th, device=dev), torch.as_tensor(r, device=dev))
                pd = A.StepPlan(A.Leapfrog(0.02), hd, zd, L_STEPS, flags=A.FLAG_ASYNC)
                for _ in range(3):
                    pd()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                for _ in range(10):
                    pd()
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / 10
                flops = 2.0 * DIM * DIM * N_CHAINS * L_STEPS
                k4 = {"workload": "C2-style: 4096 chains x D=128 correlated Gaussian (dense precision), Diag metric, L=32 fused, tiled DMMA kernel",
                      "ms_per_launch": ms, "rate_steps_dims_per_s": units_per_step / ms * 1e3, "fp64_tflops_gemm": flops / ms / 1e9}
                # the same contraction through cuBLAS Dgemm (SURVEY 8d): one [D x D] @ [D x N] product per step, 32 per
                # trajectory, as a step-at-a-time implementation would issue them; and a large Dgemm for the DMMA peak
                P64 = torch.as_tensor((Q / lam) @ Q.T, device=dev)
                X64 = torch.as_tensor(th, device=dev).T.contiguous()
                Y64 = torch.empty_like(X64)
                for _ in range(3):
                    torch.matmul(P64, X64, out=Y64)
                e0.record(stream)
                for _ in range(10 * L_STEPS):
                    torch.matmul(P64, X64, out=Y64)
                e1.record(stream)
                torch.cuda.synchronize()
                ms_cb = e0.elapsed_time(e1) / 10
                k4["cublas_dgemm_same_shape"] = {"what": "torch.matmul fp64 [128x128]@[128x4096], 32 calls = the gradient GEMMs of one trajectory (no leapfrog arithmetic)",
                                                 "ms_per_32": ms_cb, "tflops": flops / ms_cb / 1e9}
                Ab = torch.randn(4096, 4096, dtype=torch.float64, device=dev)
                Cb = torch.empty_like(Ab)
                torch.matmul(Ab, Ab, out=Cb)
                e0.record(stream)
                for _ in range(3):
                    torch.matmul(Ab, Ab, out=Cb)
                e1.record(stream)
                torch.cuda.synchronize()
                k4["cublas_dgemm_4096_tflops"] = 2.0 * 4096 ** 3 * 3 / e0.elapsed_time(e1) / 1e9
                del Ab, Cb

        # ---- fp64 FMA-pipe peak (SURVEY 8d: the bound of the fused fast path), measured by a DFMA microbenchmark
        dfma = None
        if rank == 0 and not args.no_extras:
            with Extra("dfma"):
                import ctypes
                mb = ctypes.CDLL(os.path.join(os.path.dirname(os.path.abspath(__file__)), "advancedhmc.jl_b200", "libahmc_microbench.so"))
                tf, msb = ctypes.c_double(), ctypes.c_double()
                rcmb = mb.ahmc_mb_dfma_peak(ctypes.c_int(local), ctypes.c_int(2048), ctypes.c_int(5), ctypes.byref(tf), ctypes.byref(msb))
                if rcmb == 0:
                    dfma = {"tflops": tf.value, "ms": msb.value, "what": "148*8 blocks x 256 threads x 8 independent DFMA chains (libahmc_microbench.so)"}

    # ---- the path's one exchange (SURVEY 8e), inside the driver-run line: pooled warm-up on the C4 shape (funnel D=100,
    # 4096 chains per GPU, NUTS).  Per iteration, on ONE stream and with no host synchronisation: NUTS transition (K3) ->
    # K5 record -> ncclAllGather of (2+2D) doubles per rank -> merge + dual averaging + WelfordVar + window logic in one
    # kernel that writes eps / M^-1 where the next transition reads them (ahmc_adapt_exchange_f64).  All ranks take part.
    exchange = None
    if not args.no_extras:
        with Extra("exchange"):
            from ahmc_b200 import adaptation as adp

            with torch.cuda.stream(stream):
                comm = adp.Comm.from_torch_distributed(local) if world > 1 else None
                Df, n_it = 100, 40
                hf = A.Hamiltonian(A.DiagEuclideanMetric(np.ones(Df)), A.Funnel(Df))
                gf = torch.Generator(device=dev).manual_seed(100 + rank)
                thf = 0.5 * torch.randn((N_CHAINS, Df), generator=gf, dtype=torch.float64, device=dev)
                pad = adp.PooledDeviceAdaptor(local, Df, N_CHAINS, n_adapts=n_it + 10, eps0=0.1, init_buffer=10, term_buffer=5, window_size=8)
                hdv = A.Hamiltonian(A.DiagEuclideanMetric(pad.Minv), hf.target)
                kdv = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(pad.eps), A.GeneralisedNoUTurn()))
                prf = A.PhiloxRNG(21 + rank)
                zf = A.phasepoint(hdv, thf, torch.zeros_like(thf))
                for _ in range(5):  # warm-up (also the first NCCL call)
                    trf = A.transition(prf, hdv, kdv, zf, flags=A.FLAG_ASYNC)
                    zf = trf.z
                    pad.exchange(zf.theta, trf.stat["acceptance_rate"], comm)
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nsteps_dev = torch.zeros((), dtype=torch.int64, device=dev)
                e0.record(stream)
                for _ in range(n_it):
                    trf = A.transition(prf, hdv, kdv, zf, flags=A.FLAG_ASYNC)
                    zf = trf.z
                    pad.exchange(zf.theta, trf.stat["acceptance_rate"], comm)
                    nsteps_dev += trf.stat["n_steps"].sum()
                e1.record(stream)
                torch.cuda.synchronize()
                ms_iter = e0.elapsed_time(e1) / n_it
                e0.record(stream)
                for _ in range(200):  # the exchange alone, back to back on fixed inputs
                    pad.exchange(zf.theta, trf.stat["acceptance_rate"], comm)
                e1.record(stream)
                torch.cuda.synchronize()
                us_x = e0.elapsed_time(e1) / 200 * 1e3
                tx = torch.tensor([ms_iter, us_x], dtype=torch.float64, device=dev)
                ns_all = nsteps_dev.clone()
                if world > 1:
                    dist.all_reduce(tx, op=dist.ReduceOp.MAX)
                    dist.all_reduce(ns_all)
                ms_iter_max, us_x_max = tx.tolist()
                stt = pad.state()
                exchange = {"workload": "C4 shape: Neal's funnel D=100, 4096 chains per GPU, NUTS(max_depth 10), pooled StanHMCAdaptor on the device, "
                                        f"{n_it} warm-up iterations after 5 untimed",
                            "ranks": world, "record_bytes_per_rank": (2 + 2 * Df) * 8,
                            "warmup_iteration_ms": ms_iter_max, "exchange_us": us_x_max, "exchange_share": us_x_max * 1e-3 / ms_iter_max,
                            "rate_steps_dims_per_s": float(ns_all.item()) * Df / (ms_iter_max * n_it) * 1e3,
                            "host_syncs_per_iteration": 0, "eps_after": stt["eps"],
                            "what": "exchange = K5 record + ncclAllGather + merge/adaptor kernel (ahmc_adapt_exchange_f64), max over ranks"}
                pad.destroy()
                if comm is not None:
                    comm.destroy()

    # ---- e2e: the public call with HOST (pinned) buffers, copies inside the timed region.  Contract of
    # src/integrator.jl:216-265: host arrays in (theta, r -- the cached gradient of a built-in target is recomputed on the
    # device, so it is not uploaded), a fresh phase point out (theta', r', -grad', lp', lk').  The page-locked buffers are
    # allocated with this thread bound to the GPU's NUMA node (every byte crosses PCIe; a remote node costs up to 1.5x).
    prev_affinity = A.bind_to_gpu_numa(local)
    thp = torch.as_tensor(th).pin_memory()
    rp = torch.as_tensor(r).pin_memory()
    z0h = A.PhasePoint(thp.numpy(), rp.numpy(), A.DualValue(None, None), A.DualValue(None, None))
    pin = lambda shape: torch.empty(shape, dtype=torch.float64).pin_memory()
    outs = [pin((N_CHAINS, DIM)) for _ in range(3)] + [pin((N_CHAINS,)) for _ in range(2)]
    zout = A.PhasePoint(outs[0].numpy(), outs[1].numpy(), A.DualValue(outs[3].numpy(), outs[2].numpy()),
                        A.DualValue(outs[4].numpy(), None))

    e2e_step = A.StepPlan(lf, h, z0h, L_STEPS, out=zout)

    # warm-up: the library measures its transports (zero-copy kernel loads/stores vs copy-engine pipelines of 2 / 4 chunks)
    # on the first 12 calls of a shape and keeps the fastest -- every call returns the same bytes
    for _ in range(14):
        e2e_step()
    transport = ctx.last_transport()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    call_ms = []
    import gc

    gc.collect()
    gc.disable()  # no collector pause inside a 0.3 ms call
    t0 = time.perf_counter()
    for _ in range(K):
        tc = time.perf_counter()
        ze = e2e_step()
        _ = float(ze.lp.value[0])  # device->host read of the step's result
        call_ms.append((time.perf_counter() - tc) * 1e3)
    torch.cuda.synchronize()
    gc.enable()
    e2e_mean_s = (time.perf_counter() - t0) / K
    # SURVEY 8d: "median of >= 10 reps".  The call is synchronous host code: on a shared box ONE descheduled call (62 ms was
    # observed among 0.32 ms calls) would otherwise decide the mean of 20; the mean and the extremes are reported beside it.
    e2e_s = float(np.median(call_ms)) * 1e-3 * K
    if prev_affinity is not None:
        os.sched_setaffinity(0, prev_affinity)  # the CPU arms below use every host thread again
    h2d = 2 * N_CHAINS * DIM * 8 + DIM * 8
    d2h = 3 * N_CHAINS * DIM * 8 + N_CHAINS * (8 + 8)

    # ---- reduce over ranks (max time)
    tt = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max = tt.tolist()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    value = world * units_per_step * K / (dev_ms_max * 1e-3)
    e2e_value = world * units_per_step * K / (e2e_ms_max * 1e-3)
    B = 48.0 + 24.0 / DIM  # SURVEY 8d streaming-model bytes per step*dim
    kernel_ms = dev_ms / K  # one launch per step: the event pair brackets exactly the fused kernel
    achieved = units_per_step * B / (kernel_ms * 1e-3) / 1e9
    compulsory = (N_CHAINS * DIM * 48 + N_CHAINS * 24) / (kernel_ms * 1e-3) / 1e9
    fp64_ops = units_per_step * 2 * 2  # 2 DFMA per step*dim on the fast path
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
        # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this shape, per launch, from the committed
        # `ncu --set full` capture of this round (profiles/r02/k1_headline_dram.json; null when no capture is committed)
        "traffic": measured_traffic(), "peak_source": peak_src, "kernel": "leapfrog_kernel<DIAG_GAUSS,DIAG,G=32,E=4>",
        "kernel_ms": kernel_ms,
        "model": "SURVEY 8d streaming contract: (48+24/D) B per step*dim x N*D*L units per launch; the fused L-step "
                 "kernel keeps state in registers, so its COMPULSORY traffic is 1/L of that (next keys)",
        "compulsory_bytes_per_launch": N_CHAINS * DIM * 48 + N_CHAINS * 24,
        "achieved_compulsory": compulsory, "frac_compulsory": compulsory / hbm_peak,
        "fp64_tflops_fastpath": fp64_ops / (kernel_ms * 1e-3) / 1e12,
    }
    cpu = cpu_baselines(m, s, Minv, th, r, full=True) if world == 1 else None
    line = {
        "metric": METRIC_NAME, "value": value, "unit": "steps*dims/s", "n_gpus": world, "steps": K, "warmup": max(W, 3),
        "ms_per_step": dev_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": config_dict(world),
        "roofline": roofline,
        "e2e": {"value": e2e_value, "unit": "steps*dims/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms_max / K, "ms_per_step_is": "median over the K timed calls (max over ranks); mean beside it",
                "ms_per_step_mean": e2e_mean_s * 1e3, "call_ms_min": min(call_ms), "call_ms_med": sorted(call_ms)[len(call_ms) // 2],
                "call_ms_max": max(call_ms), "transport": transport, "numa_bound": prev_affinity is not None,
                "path": "ahmc_leapfrog_f64(AHMC_FLAG_HOST_BUFFERS) via ahmc_b200.step on pinned host arrays: theta, r in; "
                        "theta', r', -grad', lp', lk' out (the cached input gradient is recomputed on the device)"},
        "gpu_launches": int(launches), "clocks": clocks,
        "step_ms_min_med_max": [float(np.min(step_ms)), float(np.median(step_ms)), float(np.max(step_ms))],
    }
    if cpu:
        line["cpu_baseline"] = {"value": cpu["numpy_1thread"], "unit": "steps*dims/s", "cores": 1, "kind": "port",
                                "sample": "full workload (4096x128x32) x3, median; numpy twin op-for-op with the reference's "
                                          "temporaries, 1 thread like Julia broadcast",
                                "omp_all_cores": {"value": cpu["omp"], "cores": cpu["cores"]}}
    if honest:
        line["roofline_hbm_honest"] = honest
    if k2:
        line["hmc_transition"] = k2
    if batch:
        roofline["launch_fixed_vs_marginal"] = batch
    if Extra.errors:
        line["extras_failed"] = Extra.errors
    if exchange:
        line["adapt_exchange"] = exchange
    if general:
        line.update(general)
    if k4:
        line["dense_target_trajectory"] = k4
    if dfma:
        line["fp64_fma_peak"] = dfma
        roofline["frac_fp64_fma_pipe"] = roofline["fp64_tflops_fastpath"] / dfma["tflops"]
        if honest and "fused_L32" in honest:
            honest["fused_L32"]["frac_fp64_fma_pipe"] = honest["fused_L32"]["fp64_tflops"] / dfma["tflops"]
    args.emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


class StdoutToStderr:
    """Native libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.
    Route fd 1 to stderr for the duration of the run and hand back a writer on the real stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.real = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.write(self.real, (text + "\n").encode())

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.real, 1)
        os.close(self.real)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    with StdoutToStderr() as out:
        args.emit = out.emit
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)


if __name__ == "__main__":
    main()
