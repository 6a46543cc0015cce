"""Cost of the pooled dense-metric adaptor on the device (K5c, dense form), in one GPU command:
    python scripts/pooled_dense_bench.py OUT_DIR [--quick]
writes OUT_DIR/pooled_dense_bench.json with the card's name and power limit read in the same run, and:
  * exchange: per ahmc_adapt_exchange_f64 call (CUDA events on the context stream, median over the calls of each kind) at
    (N, D) = (1024, 256), (4096, 128), (4096, 256), for iterations that push into a metric window and for window splits
    (which add the factorisation); and the per-kernel split -- record (K5 + K5b), pooled_cov_kernel, pooled_update_kernel,
    pooled_chol_kernel -- from a torch.profiler pass of its own (mean device time per launch);
  * cholesky: pooled_chol_kernel alone at D = 128, 256, 512 (the factorisation that creating an adaptor from Minv0 runs,
    device time from torch.profiler, median over repetitions);
  * c5_warmup: 1024 chains, D = 256, NUTS on a dense Gaussian, Minv0 = I, the same Philox streams: wall time per warm-up
    iteration of the host loop (`sample` + StanHMCAdaptor(WelfordCov): record to the host, numpy merge, host Cholesky, M^-1
    and U back to the device on every transition) against `sample_pooled_device`, each run once untimed first.
Inputs fit in L2 (at most 8.4 MB of theta); the adaptor's state lives there too, as it does in a warm-up loop."""
import json
import os
import re
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import ahmc_b200 as A
from ahmc_b200 import adaptation as ad

DEV = torch.device("cuda", 0)
KERNELS = ("adapt_kernel", "adapt_cov_kernel", "pooled_cov_kernel", "pooled_update_kernel", "pooled_chol_kernel")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[:1])


def kernel_times(prof):
    """mean device microseconds per launch and launch count of each of the adaptor's kernels"""
    out = {}
    for e in prof.key_averages():
        m = re.search(r"ahmc::(\w+)", e.key)
        if not m or m.group(1) not in KERNELS:
            continue
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        k = out.setdefault(m.group(1), dict(total_us=0.0, count=0))
        k["total_us"] += t
        k["count"] += e.count
    for k in out.values():
        k["mean_us"] = k["total_us"] / max(k["count"], 1)
    return out


def exchange_case(N, D, n_adapts, windows):
    rng = np.random.default_rng(N + D)
    Lc = np.linalg.cholesky(np.eye(D) + 0.5 * np.ones((D, D)) / D)
    th = [torch.as_tensor(rng.normal(size=(N, D)) @ Lc.T, device=DEV) for _ in range(4)]
    al = torch.as_tensor(rng.uniform(0.3, 1.0, N), device=DEV)
    ws, we, splits = ad.stan_windows(n_adapts, *windows)

    def run(timed):
        ada = ad.PooledDeviceAdaptor(0, D, N, n_adapts, 0.1, init_buffer=windows[0], term_buffer=windows[1],
                                     window_size=windows[2], dense=True)
        stream = ada.ctx.torch_stream()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_adapts)]
        torch.cuda.synchronize()
        for i in range(1, n_adapts + 1):
            if timed:
                evs[i - 1][0].record(stream)
            ada.exchange(th[i % 4], al)
            if timed:
                evs[i - 1][1].record(stream)
        torch.cuda.synchronize()
        s = ada.state()
        ada.destroy()
        assert s["failed_iteration"] == 0 and s["iteration"] == n_adapts
        return [a.elapsed_time(b) * 1e3 for a, b in evs] if timed else None

    run(False)  # warm-up: module load, the gathered / workspace buffers
    us = run(True)
    push = [us[i - 1] for i in range(ws, we + 1) if i not in splits]
    split = [us[i - 1] for i in splits if ws <= i <= we]
    outside = [us[i - 1] for i in range(1, n_adapts + 1) if not ws <= i <= we]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(False)
    k = kernel_times(prof)
    rec = sum(k.get(n, {}).get("total_us", 0.0) for n in ("adapt_kernel", "adapt_cov_kernel")) / n_adapts
    return dict(N=N, D=D, n_adapts=n_adapts, windows=list(windows), splits=splits,
                exchange_push_us_median=float(np.median(push)), exchange_split_us_median=float(np.median(split)),
                exchange_outside_window_us_median=float(np.median(outside)) if outside else None,
                per_kernel_us=dict(record_k5_k5b=rec, **{n: k[n]["mean_us"] for n in KERNELS[2:] if n in k}),
                profiler_kernels=k)


def cholesky_alone(D, reps):
    rng = np.random.default_rng(D)
    Q, _ = np.linalg.qr(rng.normal(size=(D, D)))
    M0 = (Q * np.exp(rng.uniform(0, 3, D))) @ Q.T
    M0 = (M0 + M0.T) / 2
    ad.PooledDeviceAdaptor(0, D, 64, 10, 0.1, Minv0=M0, dense=True).destroy()  # warm-up
    times = []
    for _ in range(reps):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            ada = ad.PooledDeviceAdaptor(0, D, 64, 10, 0.1, Minv0=M0, dense=True)
        s = ada.state()
        ada.destroy()
        assert np.abs(s["cholU"] - np.linalg.cholesky(M0).T).max() <= 1e-9 * np.abs(s["cholU"]).max()
        times.append(kernel_times(prof)["pooled_chol_kernel"]["mean_us"])
    return dict(D=D, reps=reps, us_median=float(np.median(times)), us_min=float(np.min(times)))


def c5_warmup(n_adapts, windows):
    D, N = 256, 1024
    rng = np.random.Generator(np.random.PCG64(11))
    Q, _ = np.linalg.qr(rng.normal(size=(D, D)))
    lam = np.exp(np.linspace(np.log(0.1), np.log(10.0), D))
    h = A.Hamiltonian(A.DenseEuclideanMetric(np.eye(D)), A.DenseGaussian(np.zeros(D), (Q / lam) @ Q.T))
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.1), A.GeneralisedNoUTurn()))
    th0 = torch.as_tensor(np.random.default_rng(1).normal(size=(N, D)), device=DEV)

    def host(n):
        adaptor = ad.StanHMCAdaptor(ad.WelfordCov(D), ad.NesterovDualAveraging(0.8, 0.1), *windows)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ad.sample(A.PhiloxRNG(5), h, kern, th0, n, adaptor=adaptor, n_adapts=n)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    def device(n):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ad.sample_pooled_device(A.PhiloxRNG(5), h, kern, th0, n, n, eps0=0.1, windows=windows)
        torch.cuda.synchronize()
        return time.perf_counter() - t0, r

    host(12)
    device(12)
    th_, rh = host(n_adapts)
    td, rd = device(n_adapts)
    return dict(N=N, D=D, n_adapts=n_adapts, windows=list(windows),
                host_loop_ms_per_iteration=th_ * 1e3 / n_adapts, device_ms_per_iteration=td * 1e3 / n_adapts,
                host_leapfrog_steps=rh.leapfrog_steps, device_leapfrog_steps=rd.leapfrog_steps,
                host_eps=rh.eps, device_eps=rd.eps,
                minv_max_abs_diff=float(np.abs(np.asarray(rh.Minv) - rd.Minv).max()))


def main():
    out_dir = sys.argv[1]
    quick = "--quick" in sys.argv
    assert torch.cuda.is_available(), "pooled_dense_bench.py measures on a GPU"
    os.makedirs(out_dir, exist_ok=True)
    res = dict(card=card())
    windows = (75, 50, 25)  # the reference's defaults: splits 100, 150, 250, 350 within 400 iterations
    n_ex = 120 if quick else 400
    res["exchange"] = [exchange_case(N, D, n_ex, windows) for N, D in ((1024, 256), (4096, 128), (4096, 256))]
    res["cholesky"] = [cholesky_alone(D, 3 if quick else 7) for D in (128, 256, 512)]
    res["c5_warmup"] = c5_warmup(30 if quick else 60, (10, 8, 6))
    res["card_after"] = card()
    path = os.path.join(out_dir, "pooled_dense_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
