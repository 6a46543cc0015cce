"""The pooled dense-metric adaptor on the device: StanHMCAdaptor(WelfordCov, NesterovDualAveraging) with the D x D merge, the
window accumulator and the Cholesky factorisation of each new M^-1 in CUDA (ahmc_pooled.cu: pooled_cov_kernel,
pooled_update_kernel, pooled_chol_kernel; ahmc_pooled_create_dense / ahmc_pooled_state_dense in the C ABI).

CPU: the kernel sources under the SIMT emulator (tests/simt_emu/pooled_dense_emu.cpp) against the host-side pooled adaptors of
adaptation.py (which tests/test_adaptation.py pins to the oracle) and numpy's Cholesky, plus a ThreadSanitizer build.
GPU: the compiled kernels against the same host adaptors, the eps-only form against the diagonal adaptor, sample_pooled_device
against the host loop, a statistical check, the error paths and (with two GPUs) an NCCL exchange."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "simt_emu")
_vp = C.c_void_p
P = lambda a: None if a is None else a.ctypes.data_as(_vp)
WINDOWS = (5, 4, 6)


def _emu_cmd(out, *extra):
    return ["g++", *extra, "-std=c++20", "-pthread", "-ffp-contract=off", "-x", "c++", "-I", os.path.join(EMU, "include"),
            "-I", os.path.join(ROOT, "advancedhmc.jl_b200", "csrc"), "-I", os.path.join(ROOT, "include"),
            os.path.join(EMU, "simt_emu.cpp"), os.path.join(EMU, "pooled_dense_emu.cpp"), "-o", str(out)]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = tmp_path_factory.mktemp("simt_pooled_dense") / "libpooled_dense_emu.so"
    pr = subprocess.run(_emu_cmd(out, "-O1", "-shared", "-fPIC"), capture_output=True, text=True)
    assert pr.returncode == 0, pr.stderr[-2000:]
    lib = C.CDLL(str(out))
    lib.emu_pd_create.restype = _vp
    lib.emu_pd_create.argtypes = [C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int,
                                  C.c_int, _vp]
    lib.emu_pd_update.argtypes = [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp]
    lib.emu_pd_destroy.argtypes = [_vp]
    lib.emu_pd_chol.argtypes = [C.c_int, _vp, _vp, _vp, C.c_int]
    return lib


def _record(th, al):
    """host layout "cov": [n, sum min(1, alpha), mean, M2diag, M2full] of one rank's (N, D) draws"""
    mu = th.mean(axis=0)
    c = th - mu
    M = c.T @ c
    M = (M + M.T) / 2  # exactly symmetric, as K5b writes it
    return np.concatenate([[th.shape[0], np.minimum(1.0, al).sum()], mu, np.diag(M).copy(), M.reshape(-1)])


def _check_factor(U, Minv, tag):
    """U upper with U'U = Minv: against numpy's factor to 1e-10 and the product to 1e-12, relative to the largest entry"""
    scale = np.abs(Minv).max()
    assert np.array_equal(U, np.triu(U)), tag
    assert np.abs(U - np.linalg.cholesky(Minv).T).max() <= 1e-10 * np.abs(U).max(), tag
    assert np.abs(U.T @ U - Minv).max() <= 1e-12 * scale, tag


def _spd(rng, D, cond=50.0):
    Q, _ = np.linalg.qr(rng.normal(size=(D, D)))
    lam = np.exp(rng.uniform(0, np.log(cond), D))
    A = (Q * lam) @ Q.T
    return (A + A.T) / 2


# ------------------------------------------------------------------------------------------------ CPU: emulated kernel sources
@pytest.mark.parametrize("R", [1, 2, 5])
@pytest.mark.parametrize("D", [1, 13, 40])
def test_dense_pooled_kernel_sources_under_emulation_equal_host_adaptors(emu, R, D):
    """K5c's dense exchange (rank-ordered D x D merge, WelfordCov push / estimate / reset, dual averaging, window schedule,
    device Cholesky at window ends) on the records R ranks with ragged chain counts would all-gather, against
    merge_records(.., "cov") + the host StanHMCAdaptor(WelfordCov) + numpy's Cholesky."""
    from ahmc_b200 import adaptation as ad

    n_adapts, eps0 = 40, 0.21
    rng = np.random.default_rng(100 * R + D)
    chains = [30 + 7 * r for r in range(R)]
    h = emu.emu_pd_create(D, chains[0], n_adapts, *WINDOWS, eps0, 0.8, 1, 3, None)
    assert h
    host = ad.StanHMCAdaptor(ad.WelfordCov(D, n_min=3), ad.NesterovDualAveraging(0.8, eps0), *WINDOWS)
    host.initialize(n_adapts)
    assert len(host.window_splits) >= 2
    Lc = np.linalg.cholesky(_spd(np.random.default_rng(D), D, 20.0))
    eps, failed = C.c_double(), C.c_int()
    minv, U, merged = np.empty(D * D), np.empty(D * D), np.empty(2 + 2 * D + D * D)
    for i in range(1, n_adapts + 1):
        recs = [_record(rng.normal(size=(chains[r], D)) @ Lc.T + 0.2 * r, rng.uniform(0.1, 1.5, chains[r])) for r in range(R)]
        gathered = np.ascontiguousarray(np.stack(recs))
        it = emu.emu_pd_update(h, P(gathered), R, C.byref(eps), P(minv), P(U), P(merged), C.byref(failed))
        assert it == i
        want = ad.merge_records(recs, "cov")
        assert np.abs(merged - want).max() <= 1e-13 * np.abs(want).max(), i
        host.adapt(want)
        if i == n_adapts:
            host.finalize()
        assert abs(eps.value - host.eps) <= 1e-13 * host.eps, (i, eps.value, host.eps)
        Mi, Ui = minv.reshape(D, D).T, U.reshape(D, D).T  # column-major buffers
        assert np.abs(Mi - host.Minv).max() <= 1e-12 * np.abs(host.Minv).max(), i
        _check_factor(Ui, Mi, i)
        assert failed.value == 0
    assert not np.array_equal(host.Minv, np.eye(D))  # the metric was adapted
    emu.emu_pd_destroy(h)


def test_dense_pooled_eps_only_under_emulation_leaves_the_metric(emu):
    """adapt_metric = 0: step size only; Minv0 and its factor stay bit for bit, the D x D record is not read"""
    from ahmc_b200 import adaptation as ad

    D, R, n_adapts = 9, 3, 30
    rng = np.random.default_rng(4)
    M0 = _spd(rng, D)
    h = emu.emu_pd_create(D, 20, n_adapts, *WINDOWS, 0.3, 0.8, 0, 3, P(np.ascontiguousarray(M0.T)))
    assert h
    host = ad.StanHMCAdaptor(ad.UnitMassMatrix(), ad.NesterovDualAveraging(0.8, 0.3), *WINDOWS)
    host.initialize(n_adapts)
    eps, failed = C.c_double(), C.c_int()
    minv, U, merged = np.empty(D * D), np.empty(D * D), np.empty(2 + 2 * D + D * D)
    for i in range(1, n_adapts + 1):
        recs = [_record(rng.normal(size=(20, D)), rng.uniform(0.1, 1.5, 20))[:2 + 2 * D] for _ in range(R)]
        assert emu.emu_pd_update(h, P(np.ascontiguousarray(np.stack(recs))), R, C.byref(eps), P(minv), P(U), P(merged),
                                 C.byref(failed)) == i
        host.adapt(ad.merge_records(recs))
        if i == n_adapts:
            host.finalize()
        assert abs(eps.value - host.eps) <= 1e-13 * host.eps
        assert np.array_equal(minv.reshape(D, D).T, M0) and not merged[2 + 2 * D:].any()
        if i == 1:
            U0 = U.copy()
        assert np.array_equal(U, U0)
    _check_factor(U0.reshape(D, D).T, M0, "Minv0")
    emu.emu_pd_destroy(h)


@pytest.mark.parametrize("D", [1, 7, 37, 40])
def test_device_cholesky_source_under_emulation_matches_numpy(emu, D):
    """pooled_chol_kernel on random SPD matrices: U against numpy, reading only the upper triangle (the strictly lower one is
    garbage here); the committed M^-1 is the candidate as given"""
    rng = np.random.default_rng(D)
    A = _spd(rng, D, 1e3)
    cand = A.copy()
    cand[np.tril_indices(D, -1)] = np.nan  # never read
    colmaj = np.ascontiguousarray(cand.T)
    minv, U = np.full(D * D, 5.0), np.full(D * D, 6.0)
    assert emu.emu_pd_chol(D, P(colmaj), P(minv), P(U), 9) == 0
    assert np.array_equal(minv, colmaj.reshape(-1), equal_nan=True)
    _check_factor(U.reshape(D, D).T, A, D)


@pytest.mark.parametrize("kind", ["indefinite", "nan-diagonal", "zero-pivot"])
def test_device_cholesky_source_under_emulation_rejects_non_spd_and_keeps_the_committed_metric(emu, kind):
    D = 12
    rng = np.random.default_rng(3)
    A = _spd(rng, D)
    if kind == "indefinite":
        A = A - 1.5 * np.linalg.eigvalsh(A).max() * np.outer(np.ones(D), np.ones(D)) / D
    elif kind == "nan-diagonal":
        A[5, 5] = np.nan
    else:
        A[0, :] = A[:, 0] = 0.0
    minv0, U0 = rng.normal(size=D * D), rng.normal(size=D * D)
    minv, U = minv0.copy(), U0.copy()
    assert emu.emu_pd_chol(D, P(np.ascontiguousarray(A.T)), P(minv), P(U), 17) == 17
    assert minv.tobytes() == minv0.tobytes() and U.tobytes() == U0.tobytes()


def test_dense_pooled_kernel_sources_are_data_race_free_under_thread_sanitizer(tmp_path):
    """the three kernels of a dense exchange (multi-block merge, update, block-barrier Cholesky) with every CUDA thread a host
    thread: a missing __syncthreads shows up as a data race"""
    out = tmp_path / "race_pooled_dense"
    pr = subprocess.run(_emu_cmd(out, "-DRACE_MAIN", "-w", "-O1", "-g", "-fsanitize=thread"), capture_output=True, text=True)
    if pr.returncode != 0 and ("tsan" in pr.stderr.lower() or "sanitize" in pr.stderr.lower()):
        pytest.skip("ThreadSanitizer runtime not available to g++ here")
    assert pr.returncode == 0, pr.stderr[-2000:]
    r = subprocess.run([str(out)], capture_output=True, text=True, timeout=600)
    if "FATAL: ThreadSanitizer" in r.stderr:
        pytest.skip("ThreadSanitizer cannot run in this environment: " + r.stderr.strip().splitlines()[0])
    assert r.stderr.count("WARNING: ThreadSanitizer: data race") == 0 and r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.count("rc 0") == 6


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda:0"


def _dev_record(A, th, al):
    D = th.shape[1]
    rec = A.adapt_summary(th, al)
    return np.concatenate([rec.cpu().numpy(), A.adapt_cov(th, rec[2:2 + D]).cpu().numpy().reshape(-1)])


@pytest.mark.gpu
@pytest.mark.parametrize("D,N,n_adapts", [(37, 300, 46), (256, 1024, 20)])
def test_device_dense_pooled_adaptor_equals_host_adaptors_iteration_by_iteration(D, N, n_adapts):
    import torch

    import ahmc_b200 as A
    from ahmc_b200 import adaptation as ad

    rng = np.random.default_rng(D)
    ada = ad.PooledDeviceAdaptor(0, D, N, n_adapts, eps0=0.13, init_buffer=WINDOWS[0], term_buffer=WINDOWS[1],
                                 window_size=WINDOWS[2], n_min=3, dense=True)
    host = ad.StanHMCAdaptor(ad.WelfordCov(D, n_min=3), ad.NesterovDualAveraging(0.8, 0.13), *WINDOWS)
    host.initialize(n_adapts)
    assert host.window_splits
    Lc = np.linalg.cholesky(_spd(rng, D, 30.0))
    trace = torch.zeros(n_adapts, dtype=torch.float64, device=DEV)
    for i in range(1, n_adapts + 1):
        th = torch.as_tensor(rng.normal(size=(N, D)) @ Lc.T + 0.3, device=DEV)
        al = torch.as_tensor(rng.uniform(0.3, 1.4, N), device=DEV)
        ada.exchange(th, al, None, trace, flags=0)
        rec = _dev_record(A, th, al)
        host.adapt(rec)
        if i == n_adapts:
            host.finalize()
        s = ada.state()
        assert s["iteration"] == i and s["failed_iteration"] == 0
        assert np.abs(s["merged_record"] - rec).max() <= 1e-13 * np.abs(rec).max(), i
        assert abs(s["eps"] - host.eps) <= 1e-12 * host.eps, (i, s["eps"], host.eps)
        assert (ada.eps.cpu().numpy() == s["eps"]).all()
        assert np.abs(s["Minv"] - host.Minv).max() <= 1e-12 * np.abs(host.Minv).max(), i
        _check_factor(s["cholU"], s["Minv"], i)
        assert np.array_equal(ada.Minv.cpu().numpy(), s["Minv"]) and np.array_equal(ada.cholU.cpu().numpy(), s["cholU"])
    assert not np.array_equal(s["Minv"], np.eye(D))
    assert trace.cpu().numpy()[-1] == s["eps"]
    ada.destroy()


@pytest.mark.gpu
def test_device_dense_pooled_adaptor_eps_only_matches_the_diagonal_adaptor_bit_for_bit():
    import torch

    from ahmc_b200 import adaptation as ad

    D, N, n_adapts = 24, 200, 40
    rng = np.random.default_rng(5)
    M0 = _spd(rng, D)
    kw = dict(eps0=0.17, adapt_metric=False, init_buffer=WINDOWS[0], term_buffer=WINDOWS[1], window_size=WINDOWS[2], n_min=3)
    dense = ad.PooledDeviceAdaptor(0, D, N, n_adapts, Minv0=M0, dense=True, **kw)
    diag = ad.PooledDeviceAdaptor(0, D, N, n_adapts, **kw)
    s0 = dense.state()
    assert np.array_equal(s0["Minv"], M0)
    _check_factor(s0["cholU"], M0, "Minv0")
    for i in range(1, n_adapts + 1):
        th = torch.as_tensor(rng.normal(size=(N, D)), device=DEV)
        al = torch.as_tensor(rng.uniform(0.3, 1.4, N), device=DEV)
        dense.exchange(th, al, flags=0)
        diag.exchange(th, al, flags=0)
        s, t = dense.state(), diag.state()
        assert s["iteration"] == t["iteration"] == i and s["eps"] == t["eps"]
        assert s["Minv"].tobytes() == s0["Minv"].tobytes() and s["cholU"].tobytes() == s0["cholU"].tobytes()
        assert not s["merged_record"][2 + 2 * D:].any()
    dense.destroy()
    diag.destroy()


def _dense_gauss(A, D, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    Q, _ = np.linalg.qr(rng.normal(size=(D, D)))
    lam = np.exp(np.linspace(np.log(0.1), np.log(10.0), D))
    Sigma, Prec = (Q * lam) @ Q.T, (Q / lam) @ Q.T
    return Sigma, A.DenseGaussian(np.zeros(D), Prec)


@pytest.mark.gpu
def test_dense_sample_pooled_device_adapts_like_the_host_loop():
    """sample_pooled_device with a DenseEuclideanMetric (cooperative dense NUTS, D = 40) against sample() with the host
    StanHMCAdaptor(WelfordCov) on the same Philox streams"""
    import torch

    import ahmc_b200 as A
    from ahmc_b200 import adaptation as ad

    D, N, n_adapts, n_samples, windows = 40, 512, 60, 70, (10, 8, 6)
    _, tgt = _dense_gauss(A, D, 21)
    h = A.Hamiltonian(A.DenseEuclideanMetric(np.eye(D)), tgt)
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.2), A.GeneralisedNoUTurn(max_depth=6)))
    th0 = torch.as_tensor(np.random.default_rng(3).normal(size=(N, D)), device=DEV)
    rd = ad.sample_pooled_device(A.PhiloxRNG(5), h, kern, th0, n_samples, n_adapts, eps0=0.2, windows=windows, keep_eps_trace=True)
    host = ad.StanHMCAdaptor(ad.WelfordCov(D), ad.NesterovDualAveraging(0.8, 0.2), *windows)
    rh = ad.sample(A.PhiloxRNG(5), h, kern, th0, n_samples, adaptor=host, n_adapts=n_adapts)
    eps_dev = np.array([st["step_size_after"] for st in rd.stats[:n_adapts]])
    eps_host = np.array([rh.stats[k + 1]["step_size"] for k in range(n_adapts - 1)] + [rh.eps])
    assert np.allclose(eps_dev[:-1], eps_host[:-1], rtol=1e-9) and abs(rd.eps - rh.eps) < 1e-9 * rh.eps
    assert rd.Minv.shape == (D, D) and np.abs(rd.Minv - rh.Minv).max() <= 1e-9 * np.abs(rh.Minv).max()
    assert not np.array_equal(rd.Minv, np.eye(D))
    assert rd.leapfrog_steps == rh.leapfrog_steps


@pytest.mark.gpu
def test_dense_sample_pooled_device_recovers_a_correlated_gaussian():
    import torch

    import ahmc_b200 as A
    from ahmc_b200 import adaptation as ad

    D, N = 32, 1024
    Sigma, tgt = _dense_gauss(A, D, 11)
    h = A.Hamiltonian(A.DenseEuclideanMetric(np.eye(D)), tgt)
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.1), A.GeneralisedNoUTurn()))
    th0 = torch.as_tensor(np.random.default_rng(1).normal(size=(N, D)), device=DEV)
    res = ad.sample_pooled_device(A.PhiloxRNG(5), h, kern, th0, 150, 150, eps0=0.1)
    assert res.Minv.shape == (D, D)
    assert np.linalg.norm(res.Minv - Sigma) / np.linalg.norm(Sigma) < 0.15
    hd = A.Hamiltonian(A.DenseEuclideanMetric(res.Minv), tgt)
    kd = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(res.eps), A.GeneralisedNoUTurn()))
    zl, draws, st = A.sample_transitions(A.PhiloxRNG(9), hd, kd, A.phasepoint(hd, res.theta, torch.zeros_like(res.theta)), 50)
    X = draws.reshape(-1, D).cpu().numpy()
    assert np.linalg.norm(np.cov(X.T) - Sigma) / np.linalg.norm(Sigma) < 0.15
    acc = st["acceptance_rate"].mean().item()
    assert 0.6 < acc < 0.97, acc


@pytest.mark.gpu
def test_dense_pooled_adaptor_errors():
    import ctypes

    import torch

    import ahmc_b200 as A
    from ahmc_b200 import _lib as L
    from ahmc_b200 import adaptation as ad

    D, N = 6, 32
    bad = np.eye(D)
    bad[2, 2] = -1.0
    with pytest.raises(L.InvalidArgument, match="not positive definite"):
        ad.PooledDeviceAdaptor(0, D, N, 20, 0.1, Minv0=bad, dense=True)
    with pytest.raises(L.AhmcError) as e:
        ad.PooledDeviceAdaptor(0, 513, N, 20, 0.1, dense=True)
    assert e.value.code == L.ERR_UNSUPPORTED
    dense = ad.PooledDeviceAdaptor(0, D, N, 20, 0.1, dense=True)
    diag = ad.PooledDeviceAdaptor(0, D, N, 20, 0.1)
    ctx = dense.ctx
    eps, it = ctypes.c_double(), ctypes.c_int32()
    assert ctx.lib.ahmc_pooled_state(ctx.h, dense.h, ctypes.byref(eps), None, ctypes.byref(it), None) == L.ERR_INVALID
    assert "ahmc_pooled_state_dense" in ctx.lib.ahmc_last_error(ctx.h).decode()
    assert ctx.lib.ahmc_pooled_state_dense(ctx.h, diag.h, None, None, None, None, None, None) == L.ERR_INVALID
    assert ctx.lib.ahmc_pooled_cholu(diag.h) is None and ctx.lib.ahmc_pooled_cholu(dense.h) is not None
    th = torch.zeros((N, D + 1), dtype=torch.float64, device=DEV)
    al = torch.ones(N, dtype=torch.float64, device=DEV)
    rc = ctx.lib.ahmc_adapt_exchange_f64(ctx.h, None, dense.h, D + 1, N, th.data_ptr(), D + 1, al.data_ptr(), None, 0)
    assert rc == L.ERR_INVALID
    dense.destroy()
    diag.destroy()


@pytest.mark.gpu
def test_dense_pooled_adaptor_keeps_the_metric_when_a_window_estimate_is_not_positive_definite():
    """one chain with a NaN coordinate pushed into the second metric window: the factorisation at that window's split fails,
    M^-1 and U keep the first window's values and failed_iteration names the split"""
    import torch

    from ahmc_b200 import adaptation as ad

    D, N, n_adapts = 13, 100, 30
    rng = np.random.default_rng(2)
    ada = ad.PooledDeviceAdaptor(0, D, N, n_adapts, 0.1, init_buffer=WINDOWS[0], term_buffer=WINDOWS[1], window_size=WINDOWS[2],
                                 n_min=3, dense=True)
    _, _, splits = ad.stan_windows(n_adapts, *WINDOWS)
    assert splits == [11, 26]
    for i in range(1, n_adapts + 1):
        x = rng.normal(size=(N, D)) * 2.0
        if i == 14:
            x[7, 4] = np.nan
        ada.exchange(torch.as_tensor(x, device=DEV), torch.as_tensor(rng.uniform(0.3, 1.0, N), device=DEV), flags=0)
        if i == 25:
            before = ada.state()
            assert before["failed_iteration"] == 0 and not np.array_equal(before["Minv"], np.eye(D))
    s = ada.state()
    assert s["failed_iteration"] == 26
    assert s["Minv"].tobytes() == before["Minv"].tobytes() and s["cholU"].tobytes() == before["cholU"].tobytes()
    ada.destroy()


@pytest.mark.gpu
def test_dense_sample_pooled_device_raises_on_a_nan_chain():
    import torch

    import ahmc_b200 as A
    from ahmc_b200 import _lib as L
    from ahmc_b200 import adaptation as ad

    D, N = 8, 64
    _, tgt = _dense_gauss(A, D, 4)
    h = A.Hamiltonian(A.DenseEuclideanMetric(np.eye(D)), tgt)
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.2), A.GeneralisedNoUTurn(max_depth=5)))
    th0 = np.random.default_rng(0).normal(size=(N, D))
    th0[3, 2] = np.nan
    first = ad.stan_windows(30, *WINDOWS)[2][0]
    with pytest.raises(L.AhmcError, match=f"iteration {first} "):
        ad.sample_pooled_device(A.PhiloxRNG(1), h, kern, torch.as_tensor(th0, device=DEV), 30, 30, eps0=0.2, windows=WINDOWS)


@pytest.mark.gpu
def test_dense_pooled_adaptor_over_nccl_two_ranks():
    """scripts/nccl_dense_exchange_check.py under torch.distributed.run: 2 ranks with ragged chain counts, eps, M^-1 and U
    bit-identical across ranks and equal to the host adaptors fed the rank-ordered merge"""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    pr = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
                         "127.0.0.1", "--master-port", "29521", os.path.join(ROOT, "scripts", "nccl_dense_exchange_check.py")],
                        capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert pr.returncode == 0 and "nccl dense exchange ok" in pr.stdout, pr.stdout[-1500:] + pr.stderr[-3000:]
