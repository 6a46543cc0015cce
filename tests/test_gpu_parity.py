"""GPU parity tests (run with -m gpu on the B200 box): the CUDA path, called through the C ABI, against
(i) the committed 50-digit known answers and (ii) the CPU oracle on the same seeded inputs.
Tolerance: 1e-10 relative fp64 (BASELINE.json north_star), written out below as TOL."""
import zlib

import numpy as np
import pytest
import torch

import ahmc_b200 as A
from oracle import oracle_c as oc
from tests.helpers import (METRIC_KINDS, MODEL_KINDS, case_arrays, golden_cases, hmc_golden_cases, nuts_golden_cases, rel_err,
                           rel_err_elem_scaled, synth_diag_gauss)

pytestmark = pytest.mark.gpu
TOL = 1e-10
GOLD = golden_cases()
DEV = "cuda:0"


def T(a):
    """(D,N) Fortran numpy -> (N,D) contiguous cuda tensor (same bytes)."""
    return torch.as_tensor(np.ascontiguousarray(np.asarray(a).T), dtype=torch.float64, device=DEV)


def F(t):
    """(N,D) tensor / ndarray -> (D,N) numpy view for comparison with the oracle."""
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    return a.T if a.ndim == 2 else a


def make_target(kind, D, p0, p1, c0):
    if kind == "std_normal":
        return A.StdNormal(D, c0)
    if kind == "diag_gauss":
        t = A.DiagGaussian(p0, p1, normalised=False)
        t.c0 = c0
        return t
    if kind == "dense_gauss":
        return A.DenseGaussian(p0, p1, c0)
    return A.Funnel(D, c0)


def make_metric(kind, Minv, D):
    if kind == "unit":
        return A.UnitEuclideanMetric(D)
    if kind == "diag":
        Mi = np.asarray(Minv)
        return A.DiagEuclideanMetric(np.ascontiguousarray(Mi.T) if Mi.ndim == 2 else Mi)
    return A.DenseEuclideanMetric(np.asarray(Minv))


def assert_pp_close(z, ref, tol=TOL, fields=("theta", "r", "lp_gradient", "lp_value", "lk_value")):
    got = dict(theta=F(z.theta), r=F(z.r), lp_gradient=F(z.lp.gradient), lp_value=F(z.lp.value), lk_value=F(z.lk.value))
    if z.lk.gradient is not None:
        got["lk_gradient"] = F(z.lk.gradient)
    for f in fields:
        want = ref[f] if isinstance(ref, dict) else getattr(ref, f)
        assert rel_err(got[f], want) < tol, (f, rel_err(got[f], want))
        # element-wise: every coordinate carries its own digits (floor: 1e-3 of the largest coordinate)
        assert rel_err_elem_scaled(got[f], want) < 10 * tol, (f, "element-wise", rel_err_elem_scaled(got[f], want))


# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", GOLD["cases"], ids=[c["name"] for c in GOLD["cases"]])
@pytest.mark.parametrize("exact", [False, True], ids=["auto", "exact_checks"])
def test_leapfrog_matches_mp50_golden(case, exact):
    a = case_arrays(case)
    D = case["D"]
    h = A.Hamiltonian(make_metric(case["metric"], a["Minv"], D), make_target(case["model"], D, a["p0"], a["p1"], case["c0"]))
    z0 = A.phasepoint(h, T(a["theta0"]), T(a["r0"]))
    eps = a["eps"] if np.ndim(a["eps"]) == 0 else torch.as_tensor(a["eps"], device=DEV)
    lf = A.TemperedLeapfrog(eps, case["temper_alpha"]) if case["temper_alpha"] else A.Leapfrog(eps)
    z1, info = A.step(lf, h, z0, case["n_steps"], flags=A.FLAG_EXACT_CHECKS if exact else 0, return_info=True)
    assert (info.status == 0).all() and (info.steps_done == abs(case["n_steps"])).all()
    assert_pp_close(z1, a)


LAYOUT_DS = [1, 3, 4, 5, 8, 10, 16, 17, 32, 33, 64, 100, 128, 129, 200, 256, 300, 512]


@pytest.mark.parametrize("D", LAYOUT_DS)
def test_every_register_layout_diag(D):
    """all (G,E) layouts, ragged N (not a multiple of chains-per-block), per-chain eps, fast path."""
    rng = np.random.default_rng(D)
    N = 37
    s = np.exp(rng.uniform(-1, 1, D))
    m = rng.normal(size=D)
    Minv = np.exp(rng.uniform(-1, 1, D))
    th, r = rng.normal(size=(D, N)), rng.normal(size=(D, N))
    eps = 0.05 * np.exp(rng.uniform(-0.3, 0.3, N))
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s, 0.25), oc.Metric(oc.DIAG, Minv)
    zo, _, _ = oc.leapfrog(om, ome, eps, oc.phasepoint(om, ome, th, r), 13)
    tgt = A.DiagGaussian(m, s, normalised=False)
    tgt.c0 = 0.25
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), tgt)
    z0 = A.phasepoint(h, T(th), T(r))
    z1 = A.step(A.Leapfrog(torch.as_tensor(eps, device=DEV)), h, z0, 13)
    assert_pp_close(z1, zo, fields=("theta", "r", "lp_gradient", "lp_value", "lk_value", "lk_gradient"))


MODELS = ["std_normal", "diag_gauss", "dense_gauss", "funnel"]
METRICS = ["unit", "diag", "diag_perchain", "dense"]


@pytest.mark.parametrize("model", MODELS)
@pytest.mark.parametrize("metric", METRICS)
@pytest.mark.parametrize("D,n_steps", [(6, 9), (40, -7), (130, 5)])
def test_model_metric_matrix_vs_oracle(model, metric, D, n_steps):
    rng = np.random.default_rng(zlib.crc32(f"{model}/{metric}/{D}".encode()))  # a fixed seed per case (str hashes vary per process)
    N = 11
    p0 = p1 = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.7, 0.7, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    Minv = None
    mk = "diag" if metric == "diag_perchain" else metric
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.7, 0.7, D))
    elif metric == "diag_perchain":
        Minv = np.exp(rng.uniform(-0.7, 0.7, (D, N)))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    scale = 0.3 if model == "funnel" else 1.0
    th, r = rng.normal(size=(D, N)) * scale, rng.normal(size=(D, N))
    eps = 0.04
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.5), oc.Metric(METRIC_KINDS[mk], Minv)
    z0o = oc.phasepoint(om, ome, th, r)
    zo, st_o, dn_o = oc.leapfrog(om, ome, eps, z0o, n_steps)
    h = A.Hamiltonian(make_metric(mk, Minv, D), make_target(model, D, p0, p1, 0.5))
    z0 = A.phasepoint(h, T(th), T(r))
    assert_pp_close(z0, z0o, tol=1e-12, fields=("lp_gradient", "lp_value", "lk_value", "lk_gradient"))
    z1, info = A.step(A.Leapfrog(eps), h, z0, n_steps, return_info=True)
    assert (F(info.steps_done) == dn_o).all()
    assert_pp_close(z1, zo, fields=("theta", "r", "lp_gradient", "lp_value", "lk_value", "lk_gradient"))


def test_host_buffer_call_equals_device_call():
    D, N = 128, 257
    m, s, Minv, th, r = synth_diag_gauss(D, N, 7)
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s))
    zd = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, T(th), T(r)), 32)
    thh, rh = np.ascontiguousarray(th.T), np.ascontiguousarray(r.T)
    zh = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, thh, rh), 32)
    assert isinstance(zh.theta, np.ndarray)
    for a, b in [(zh.theta, zd.theta), (zh.r, zd.r), (zh.lp.value, zd.lp.value), (zh.lk.value, zd.lk.value),
                 (zh.lp.gradient, zd.lp.gradient), (zh.lk.gradient, zd.lk.gradient)]:
        assert np.array_equal(a, b.cpu().numpy())


def test_fast_path_equals_exact_path_within_tol_and_headline_shape_vs_oracle():
    """BASELINE headline shape: 4096 chains x D=128 diagonal Gaussian, Diag metric, eps=0.1, L=32."""
    D, N = 128, 4096
    m, s, Minv, th, r = synth_diag_gauss(D, N, 20260923)
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s))
    z0 = A.phasepoint(h, T(th), T(r))
    zf = A.step(A.Leapfrog(0.1), h, z0, 32)
    ze = A.step(A.Leapfrog(0.1), h, z0, 32, flags=A.FLAG_EXACT_CHECKS)
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s, h.target.c0), oc.Metric(oc.DIAG, Minv)
    zo, _, _ = oc.leapfrog(om, ome, 0.1, oc.phasepoint(om, ome, th, r), 32)
    assert_pp_close(zf, zo)
    assert_pp_close(ze, zo)
    assert rel_err(F(zf.theta), F(ze.theta)) < 1e-12


def test_nonfinite_per_chain_freeze_and_compat_break_all():
    """integrator.jl:252-258, hamiltonian.jl:95-104,141-142, quirk Q1."""
    D, N = 3, 6
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.StdNormal(D))
    th = np.ones((D, N))
    th[:, 2] = 1e200
    th[1, 4] = np.inf
    r = np.ones((D, N))
    om, ome = oc.Model(oc.STD_NORMAL, D), oc.Metric(oc.UNIT)
    z0o = oc.phasepoint(om, ome, th, r)
    z0 = A.phasepoint(h, T(th), T(r))
    assert F(z0.lp.value)[2] == -np.inf and F(z0.lp.value)[4] == -np.inf
    for compat in (False, True):
        zo, st_o, dn_o = oc.leapfrog(om, ome, 0.1, z0o, 5, compat_break_all=compat)
        z1, info = A.step(A.Leapfrog(0.1), h, z0, 5, flags=A.FLAG_COMPAT_BREAK_ALL if compat else 0, return_info=True)
        assert (F(info.steps_done) == dn_o).all(), (compat, F(info.steps_done), dn_o)
        assert (F(info.status) == st_o).all()
        ok = [0, 1, 3, 5]
        assert rel_err(F(z1.theta)[:, ok], zo.theta[:, ok]) < TOL
        assert F(z1.lp.value)[2] == -np.inf and F(z1.lk.value)[2] == zo.lk_value[2]
        assert np.array_equal(np.isnan(F(z1.theta)), np.isnan(zo.theta))


def test_fast_path_falls_back_to_exact_on_huge_values():
    """A chain that leaves the magnitude-proof range is re-run by the exact path in the same launch."""
    D, N = 128, 9
    m, s, Minv, th, r = synth_diag_gauss(D, N, 3)
    th[5, 3] = 1e250  # finite, but its square overflows: non-finite energy at step 1
    th[7, 6] = 1e120  # large but every energy stays finite: must complete all steps
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s), oc.Metric(oc.DIAG, Minv)
    zo, st_o, dn_o = oc.leapfrog(om, ome, 0.1, oc.phasepoint(om, ome, th, r), 20)
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s, normalised=False))
    z1, info = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, T(th), T(r)), 20, return_info=True)
    assert list(dn_o) == list(F(info.steps_done)) and dn_o[3] == 1 and dn_o[6] == 20
    assert (F(info.status) == st_o).all()
    ok = [c for c in range(N) if c != 3]
    assert rel_err(F(z1.theta)[:, ok], zo.theta[:, ok]) < TOL and rel_err(F(z1.r)[:, ok], zo.r[:, ok]) < TOL
    assert rel_err(F(z1.lk.value)[ok], zo.lk_value[ok]) < TOL


def test_in_place_and_zero_steps_and_empty():
    D, N = 10, 64
    rng = np.random.default_rng(0)
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.StdNormal(D))
    z0 = A.phasepoint(h, T(rng.normal(size=(D, N))), T(rng.normal(size=(D, N))))
    ref = A.step(A.Leapfrog(0.1), h, z0, 32)
    same = A.step(A.Leapfrog(0.1), h, z0, 0)
    assert torch.equal(same.theta, z0.theta) and torch.equal(same.lp.value, z0.lp.value)
    # in place through the raw ABI: z_out == z_in
    import ctypes as C

    ctx = A.get_context(0)
    zc = z0._c()
    md, _ = h.metric._desc(D, N, z0.theta)
    ctx.check(ctx.lib.ahmc_leapfrog_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, 0.1, None, 32, 0.0,
                                        C.byref(zc), C.byref(zc), None, None, 0))
    assert torch.equal(z0.theta, ref.theta) and torch.equal(z0.r, ref.r) and torch.equal(z0.lk.value, ref.lk.value)
    # N = 0 is a no-op
    e = torch.empty((0, D), dtype=torch.float64, device=DEV)
    ze = A.phasepoint(h, e, e.clone())
    assert A.step(A.Leapfrog(0.1), h, ze, 3).theta.shape == (0, D)


def test_argument_errors_like_the_reference():
    """ArgumentError analogues (hamiltonian.jl:53-57, :94)."""
    D, N = 5, 4
    h = A.Hamiltonian(A.DiagEuclideanMetric(np.ones(D + 1)), A.StdNormal(D))
    th = torch.zeros((N, D), dtype=torch.float64, device=DEV)
    with pytest.raises(ValueError, match="AxesMismatch"):
        A.phasepoint(h, th, th.clone())
    h2 = A.Hamiltonian(A.UnitEuclideanMetric(D), A.StdNormal(D + 2))
    with pytest.raises(ValueError, match="AxesMismatch"):
        A.phasepoint(h2, th, th.clone())
    with pytest.raises(ValueError):
        A.phasepoint(A.Hamiltonian(A.UnitEuclideanMetric(D), A.StdNormal(D)), th, torch.zeros((N, D + 1), dtype=torch.float64, device=DEV))
    big = torch.zeros((2, 513), dtype=torch.float64, device=DEV)
    with pytest.raises(A.AhmcError, match="register-resident"):  # beyond 512 dimensions only the streaming combinations exist
        A.phasepoint(A.Hamiltonian(A.DenseEuclideanMetric(np.eye(513)), A.StdNormal(513)), big, big.clone())


# ------------------------------------------------------------------------------------------------ properties at scale
def test_full_size_properties():
    """Size-independent properties at 2^17 chains x D=128 (no oracle run needed):
    reversibility, chain independence / permutation equivariance, energy error O(eps^2)."""
    D, N = 128, 1 << 17
    g = torch.Generator(device=DEV).manual_seed(1)
    s = torch.exp(torch.linspace(np.log(0.1), np.log(10.0), D, dtype=torch.float64, device=DEV))
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.DiagGaussian(np.zeros(D), s.cpu().numpy()))
    th = torch.randn((N, D), generator=g, dtype=torch.float64, device=DEV) * s
    r = torch.randn((N, D), generator=g, dtype=torch.float64, device=DEV) / s
    z0 = A.phasepoint(h, th, r)
    z1 = A.step(A.Leapfrog(0.1), h, z0, 32)
    zb = A.step(A.Leapfrog(0.1), h, z1, -32)
    assert ((zb.theta - th).abs().max() / th.abs().max()).item() < 1e-12
    assert ((zb.r - r).abs().max() / r.abs().max()).item() < 1e-12
    dH = (A.energy(z1) - A.energy(z0)).abs().max().item()
    assert dH < 0.5 * D  # leapfrog at eps=0.1 on unit-frequency modes: bounded energy error
    perm = torch.randperm(N, device=DEV, generator=g)
    zp = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, th[perm].contiguous(), r[perm].contiguous()), 32)
    assert torch.equal(zp.theta, z1.theta[perm]) and torch.equal(zp.lk.value, z1.lk.value[perm])
    # 32 x step(1) == step(32) within rounding (test/integrator.jl:17-32, there atol 5e-3)
    zl = z0
    for _ in range(4):
        zl = A.step(A.Leapfrog(0.1), h, zl, 8)
    assert ((zl.theta - z1.theta).abs().max() / z1.theta.abs().max()).item() < 1e-12


# ------------------------------------------------------------------------------------------------ transitions
@pytest.mark.parametrize("model,metric,D", [("diag_gauss", "diag", 128), ("std_normal", "unit", 10),
                                            ("funnel", "diag", 20), ("dense_gauss", "dense", 12)])
def test_hmc_transition_vs_oracle_with_tapes(model, metric, D):
    rng = np.random.default_rng(D)
    N = 301
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.5, 0.5, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    th = rng.normal(size=(D, N)) * (0.3 if model == "funnel" else 1.0)
    nt, et = rng.normal(size=(D, N)), rng.exponential(size=N) * 0.02
    eps, L = {"diag_gauss": (0.6, 10), "std_normal": (0.9, 10), "funnel": (0.1, 8), "dense_gauss": (0.3, 10)}[model]
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.0), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, np.zeros((D, N)))
    zo, so = oc.hmc_transition(om, ome, eps, L, z0o, nt, et)
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.0))
    z0 = A.phasepoint(h, T(th), T(np.zeros((D, N))))
    tau = A.Trajectory(A.EndPointTS, A.Leapfrog(eps), A.FixedNSteps(L))
    tr = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(et, device=DEV)), h, A.HMCKernel(tau), z0)
    acc = F(tr.stat["is_accept"]).astype(bool)
    assert 0 < acc.sum() < N
    assert (acc == so.is_accept.astype(bool)).all()
    assert_pp_close(tr.z, zo)
    assert rel_err(F(tr.stat["acceptance_rate"]), so.acceptance_rate) < 1e-9
    assert np.allclose(F(tr.stat["hamiltonian_energy_error"]), so.hamiltonian_energy_error, rtol=0, atol=1e-9 * D)
    assert rel_err(F(tr.stat["hamiltonian_energy"]), so.hamiltonian_energy) < TOL
    assert (F(tr.stat["n_steps"]) == L).all() and (F(tr.stat["numerical_error"]) == so.numerical_error).all()
    assert tr.stat["step_size"] == eps and tr.stat["nom_step_size"] == eps


def test_rand_momentum_tape_and_philox_moments():
    D, N = 6, 50_000
    rng = np.random.default_rng(0)
    B = rng.normal(size=(D, D))
    Minv = B @ B.T / D + 0.5 * np.eye(D)
    nt = rng.normal(size=(D, 64))
    for me_o, me in [(oc.Metric(oc.UNIT), A.UnitEuclideanMetric(D)), (oc.Metric(oc.DIAG, np.diag(Minv).copy()), A.DiagEuclideanMetric(np.diag(Minv).copy())),
                     (oc.Metric(oc.DENSE, Minv), A.DenseEuclideanMetric(Minv))]:
        got = F(A.rand_momentum(A.TapeRNG(normal=T(nt)), me, None, T(nt)))
        want = np.stack([_orc_rand_momentum(me_o, nt[:, c]) for c in range(64)], axis=1)
        assert rel_err(got, want) < 1e-12
    # Philox: r ~ N(0, M) with M = inv(Minv)   (metric.jl:311-320 => cov(r) = M)
    th = torch.zeros((N, D), dtype=torch.float64, device=DEV)
    r = A.rand_momentum(A.PhiloxRNG(123), A.DenseEuclideanMetric(Minv), None, th).cpu().numpy()
    M = np.linalg.inv(Minv)
    assert np.abs(r.mean(axis=0)).max() < 5 * np.sqrt(np.diag(M).max() / N)
    assert np.abs(np.cov(r.T) - M).max() < 0.05 * np.abs(M).max()
    r2 = A.rand_momentum(A.PhiloxRNG(123), A.DenseEuclideanMetric(Minv), None, th).cpu().numpy()
    assert np.array_equal(r, r2)  # counter-based: same (seed, offset) -> same draw
    # identical per-chain generators are impossible by construction (chain index is in the counter):
    assert len({tuple(x) for x in r[:100]}) == 100


def _orc_rand_momentum(me, z):
    import ctypes as C

    r = np.zeros_like(z)
    z = np.ascontiguousarray(z)
    oc.lib().orc_rand_momentum(C.byref(me.c), C.c_int32(z.size), C.c_int64(0), z.ctypes.data_as(oc._dp), r.ctypes.data_as(oc._dp))
    return r


def test_hmc_sampling_moments_philox():
    """test/sampler-vec.jl:43 analogue: many chains, Philox randomness, mean ~ target mean."""
    D, N = 5, 4096
    m, s = np.array([1.0, -2.0, 0.5, 0.0, 3.0]), np.array([1.0, 0.5, 2.0, 1.5, 0.7])
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.DiagGaussian(m, s))
    z = A.phasepoint(h, torch.zeros((N, D), dtype=torch.float64, device=DEV), torch.zeros((N, D), dtype=torch.float64, device=DEV))
    kern = A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.2), A.FixedNSteps(10)))
    rng = A.PhiloxRNG(2026)
    acc = 0.0
    for _ in range(60):
        tr = A.transition(rng, h, kern, z)
        z = tr.z
        acc += tr.stat["acceptance_rate"].mean().item()
    th = z.theta.cpu().numpy()
    assert np.abs(th.mean(axis=0) - m).max() < 0.15 and np.abs(th.std(axis=0) - s).max() < 0.15
    assert 0.6 < acc / 60 <= 1.0


def test_adapt_summary_matches_numpy():
    D, N = 100, 4097
    rng = np.random.default_rng(1)
    th = rng.normal(size=(N, D)) * 3 + 1
    al = rng.uniform(0, 1.4, N)
    out = A.adapt_summary(torch.as_tensor(th, device=DEV), torch.as_tensor(al, device=DEV)).cpu().numpy()
    assert out[0] == N and out[1] == pytest.approx(np.minimum(1, al).sum(), rel=1e-13)
    assert np.allclose(out[2:2 + D], th.mean(axis=0), rtol=1e-12)
    assert np.allclose(out[2 + D:], ((th - th.mean(axis=0)) ** 2).sum(axis=0), rtol=1e-12)
    out2 = A.adapt_summary(torch.as_tensor(th, device=DEV), torch.as_tensor(al, device=DEV)).cpu().numpy()
    assert np.array_equal(out, out2)  # deterministic reduction order


@pytest.mark.parametrize("D,N", [(7, 33), (100, 4097), (256, 1024), (33, 5)])
def test_adapt_cov_matches_numpy(D, N):
    """K5b (ahmc_adapt_cov_f64): full second-moment matrix about the K5 mean, symmetric, deterministic; host buffers too."""
    rng = np.random.default_rng(D)
    Lm = rng.normal(size=(D, D)) / np.sqrt(D)
    th = rng.normal(size=(N, D)) @ Lm + rng.normal(size=D)
    tht = torch.as_tensor(th, device=DEV)
    rec = A.adapt_summary(tht, None)
    out = A.adapt_cov(tht, rec[2:2 + D]).cpu().numpy()
    c = th - th.mean(axis=0)
    want = c.T @ c
    assert np.allclose(out, want, rtol=1e-11, atol=1e-11 * np.abs(want).max())
    assert np.array_equal(out, out.T)
    assert np.array_equal(out, A.adapt_cov(tht, rec[2:2 + D]).cpu().numpy())
    assert np.allclose(np.diag(out), rec[2 + D:].cpu().numpy(), rtol=1e-11)
    outh = A.adapt_cov(th, th.mean(axis=0))
    assert np.allclose(outh, want, rtol=1e-11, atol=1e-11 * np.abs(want).max())


# ------------------------------------------------------------------------------------------------ NUTS
_SAMPLERS = {"multinomial": "MultinomialTS", "slice": "SliceTS"}
_CRITERIA = {"generalised": "GeneralisedNoUTurn", "classic": "ClassicNoUTurn", "strict": "StrictGeneralisedNoUTurn"}


def _nuts_case(model, metric, D, N, eps, seed, max_depth=10, scale=1.0, sampler="multinomial", criterion="generalised"):
    rng = np.random.default_rng(seed)
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.5, 0.5, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    th = rng.normal(size=(D, N)) * scale
    nt = rng.normal(size=(D, N))
    dirs = rng.integers(0, 2, size=(N, max_depth + 1)).astype(np.uint8)
    exps = rng.exponential(size=(N, 1 << max_depth))
    if sampler == "slice":  # SliceTS: one randexp for the slice variable, then rand() uniforms (trajectory.jl:144-145, 178-183, 202)
        exps[:, 1:] = rng.uniform(size=(N, (1 << max_depth) - 1))
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.0), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, np.zeros((D, N)))
    zo, so, used = oc.nuts_transition(om, ome, eps, z0o, nt, dirs, exps, max_depth=max_depth, sampler=sampler,
                                      criterion=criterion)
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.0))
    z0 = A.phasepoint(h, T(th), T(np.zeros((D, N))))
    tau = A.Trajectory(getattr(A, _SAMPLERS[sampler]), A.Leapfrog(eps), getattr(A, _CRITERIA[criterion])(max_depth, 1000.0))
    rngt = A.TapeRNG(normal=T(nt), exp=torch.as_tensor(exps, device=DEV), dirs=torch.as_tensor(dirs, device=DEV))
    tr = A.transition(rngt, h, A.HMCKernel(tau), z0)
    return tr, zo, so


@pytest.mark.parametrize("model,metric,D,eps,scale", [
    ("std_normal", "unit", 10, 0.3, 1.0), ("diag_gauss", "diag", 128, 0.15, 1.0), ("diag_gauss", "unit", 5, 0.4, 1.0),
    ("funnel", "diag", 20, 0.12, 0.6), ("dense_gauss", "dense", 12, 0.25, 1.0), ("diag_gauss", "diag", 200, 0.1, 1.0),
    ("funnel", "unit", 3, 0.9, 2.0),
    ("funnel", "diag", 100, 0.1, 0.5),        # BASELINE C4's own shape
    ("dense_gauss", "dense", 256, 0.2, 1.0),  # BASELINE C5's own shape: E = 8 layout, level slots cache M^-1 r_first
])
def test_nuts_transition_vs_oracle_with_tapes(model, metric, D, eps, scale):
    N = 203 if D < 256 else 48
    tr, zo, so = _nuts_case(model, metric, D, N, eps, seed=D * 7 + 1, scale=scale)
    st = tr.stat
    assert (F(st["tree_depth"]) == so.tree_depth).all(), (F(st["tree_depth"])[:20], so.tree_depth[:20])
    assert (F(st["n_steps"]) == so.n_steps).all()
    assert (F(st["numerical_error"]) == so.numerical_error).all()
    if D <= 32:
        assert len(set(so.tree_depth)) > 1  # several chains per warp with divergent tree sizes
    assert_pp_close(tr.z, zo)
    assert rel_err(F(st["acceptance_rate"]), so.acceptance_rate) < 1e-9
    assert np.allclose(F(st["hamiltonian_energy_error"]), so.hamiltonian_energy_error, rtol=0, atol=1e-9 * D)
    assert np.allclose(F(st["max_hamiltonian_energy_error"]), so.max_hamiltonian_energy_error, rtol=1e-6, atol=1e-9 * D)
    assert (F(st["is_accept"]) == 1).all()


@pytest.mark.parametrize("sampler,criterion", [
    ("slice", "generalised"), ("multinomial", "classic"), ("multinomial", "strict"), ("slice", "classic"), ("slice", "strict"),
])
@pytest.mark.parametrize("model,metric,D,eps,scale", [
    ("std_normal", "unit", 10, 0.3, 1.0), ("diag_gauss", "diag", 128, 0.15, 1.0), ("funnel", "diag", 20, 0.12, 0.6),
    ("dense_gauss", "dense", 12, 0.25, 1.0), ("funnel", "unit", 3, 0.9, 2.0),
])
def test_nuts_variants_vs_oracle_with_tapes(sampler, criterion, model, metric, D, eps, scale):
    """SliceTS / ClassicNoUTurn / StrictGeneralisedNoUTurn (trajectory.jl:102-109, 551-557, 579-613): same trees,
    same draws and same statistics as the oracle, chain by chain, from shared random tapes."""
    N = 203
    tr, zo, so = _nuts_case(model, metric, D, N, eps, seed=D * 11 + 3, scale=scale, sampler=sampler, criterion=criterion)
    st = tr.stat
    assert (F(st["tree_depth"]) == so.tree_depth).all(), (F(st["tree_depth"])[:20], so.tree_depth[:20])
    assert (F(st["n_steps"]) == so.n_steps).all()
    assert (F(st["numerical_error"]) == so.numerical_error).all()
    assert_pp_close(tr.z, zo)
    assert rel_err(F(st["acceptance_rate"]), so.acceptance_rate) < 1e-9
    assert np.allclose(F(st["hamiltonian_energy_error"]), so.hamiltonian_energy_error, rtol=0, atol=1e-9 * D)
    assert np.allclose(F(st["max_hamiltonian_energy_error"]), so.max_hamiltonian_energy_error, rtol=1e-6, atol=1e-9 * D)


def test_nuts_variants_differ_from_default_and_sample_the_target():
    """the criteria are not aliases of each other (tree sizes differ on an anisotropic target), and SliceTS +
    ClassicNoUTurn with Philox randomness still recovers the target moments."""
    tr_g, _, so_g = _nuts_case("diag_gauss", "unit", 16, 256, 0.2, seed=77)
    tr_c, _, so_c = _nuts_case("diag_gauss", "unit", 16, 256, 0.2, seed=77, criterion="classic")
    tr_s, _, so_s = _nuts_case("diag_gauss", "unit", 16, 256, 0.2, seed=77, criterion="strict")
    assert (F(tr_g.stat["n_steps"]) != F(tr_c.stat["n_steps"])).any()
    assert (F(tr_s.stat["n_steps"]) <= F(tr_g.stat["n_steps"])).all()  # strict adds checks: never a larger tree
    D, N = 6, 2048
    m, s = np.linspace(-2, 2, D), np.exp(np.linspace(-1, 1, D))
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.DiagGaussian(m, s))
    kern = A.HMCKernel(A.Trajectory(A.SliceTS, A.Leapfrog(0.5), A.ClassicNoUTurn()))
    z = A.phasepoint(h, T(np.zeros((D, N))), T(np.zeros((D, N))))
    zl, draws, st = A.sample_transitions(A.PhiloxRNG(11), h, kern, z, 60)
    x = draws[20:].reshape(-1, D).cpu().numpy()
    assert np.abs(x.mean(0) - m).max() < 0.05 * s.max()
    assert np.abs(x.std(0) / s - 1).max() < 0.05
    with pytest.raises(A.AhmcError):
        A.transition(A.PhiloxRNG(0), h, A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.1), A.ClassicNoUTurn())), z)


_HMC_GOLD = hmc_golden_cases()


@pytest.mark.parametrize("case", _HMC_GOLD, ids=[c["name"] for c in _HMC_GOLD])
def test_static_transitions_match_mp50_restatement(case):
    """K2 (refresh + trajectory + Metropolis step + flip) and the MultinomialTS static kernel through the C ABI against
    tests/golden/hmc_mp50.json (50-digit restatement of metric.jl:290-320 and trajectory.jl:271-390)."""
    D, N = case["D"], case["N"]
    p0 = None if case["p0"] is None else np.array(case["p0"])
    p1 = None if case["p1"] is None else np.array(case["p1"])
    Minv = None if case["Minv"] is None else np.array(case["Minv"])
    h = A.Hamiltonian(make_metric(case["metric"], Minv, D), make_target(case["model"], D, p0, p1, case["c0"]))
    th0 = torch.as_tensor(np.array(case["theta0"]), device=DEV)
    z0 = A.phasepoint(h, th0, torch.zeros_like(th0))
    normals = torch.as_tensor(np.array(case["normals"]), device=DEV)
    var = torch.as_tensor(np.array(case["variates"]), device=DEV)
    alpha = case.get("temper_alpha", 0.0)  # > 0: the case's integrator is TemperedLeapfrog(eps, alpha)
    lf = A.TemperedLeapfrog(case["eps"], alpha) if alpha > 0 else A.Leapfrog(case["eps"])
    if case["sampler"] == "endpoint":
        tau = A.Trajectory(A.EndPointTS, lf, A.FixedNSteps(case["n_steps"]))
        tr = A.transition(A.TapeRNG(normal=normals, exp=var), h, A.HMCKernel(tau), z0)
    else:
        tau = A.Trajectory(A.MultinomialTS, lf, A.FixedNSteps(case["n_steps"]))
        tr = A.transition(A.TapeRNG(normal=normals, exp=var, n_fwd=case["n_fwd"]), h, A.HMCKernel(tau), z0)
        if "index" in case["expect"]:  # (the reference does not report the drawn index: absent in reference-generated cases)
            assert (tr.stat["tree_depth"].cpu().numpy() == np.array(case["expect"]["index"])).all()
    e, st, z = case["expect"], tr.stat, tr.z
    assert (st["is_accept"].cpu().numpy().astype(bool) == np.array(e["is_accept"])).all()
    for got, want in ((z.theta, e["theta"]), (z.r, e["r"]), (z.lp.gradient, e["lp_gradient"])):
        assert rel_err(got.cpu().numpy(), np.array(want)) < TOL
    assert np.allclose(z.lp.value.cpu().numpy(), e["lp_value"], rtol=1e-10, atol=1e-10)
    assert np.allclose(z.lk.value.cpu().numpy(), e["lk_value"], rtol=1e-10, atol=1e-10)
    assert np.allclose(st["acceptance_rate"].cpu().numpy(), e["acceptance_rate"], rtol=1e-10)
    assert np.allclose(st["hamiltonian_energy_error"].cpu().numpy(), e["hamiltonian_energy_error"], rtol=1e-9, atol=1e-10)


_NUTS_GOLD = nuts_golden_cases()


@pytest.mark.parametrize("case", _NUTS_GOLD, ids=[c["name"] for c in _NUTS_GOLD])
def test_nuts_kernel_matches_mp50_recursive_restatement(case):
    """K3 through the C ABI against tests/golden/nuts_mp50.json (recursive 50-digit restatement of
    src/trajectory.jl:626-742, independent of the C oracle): identical trees and selections, outputs to 1e-10."""
    D, N = case["D"], case["N"]
    p0 = None if case["p0"] is None else np.array(case["p0"])
    p1 = None if case["p1"] is None else np.array(case["p1"])
    Minv = None if case["Minv"] is None else np.array(case["Minv"])
    h = A.Hamiltonian(make_metric(case["metric"], Minv, D), make_target(case["model"], D, p0, p1, case["c0"]))
    z0 = A.phasepoint(h, torch.as_tensor(np.array(case["theta0"]), device=DEV), torch.as_tensor(np.array(case["r0"]), device=DEV))
    alpha = case.get("temper_alpha", 0.0)  # > 0: the case's integrator is TemperedLeapfrog(eps, alpha)
    lf = A.TemperedLeapfrog(case["eps"], alpha) if alpha > 0 else A.Leapfrog(case["eps"])
    tau = A.Trajectory(getattr(A, _SAMPLERS[case["sampler"]]), lf,
                       getattr(A, _CRITERIA[case["criterion"]])(case["max_depth"], case["delta_max"]))
    rngt = A.TapeRNG(exp=torch.as_tensor(np.array(case["variates"]), device=DEV),
                     dirs=torch.as_tensor(np.array(case["dirs"], dtype=np.uint8), device=DEV))
    tr = A.transition(rngt, h, tau, z0)  # a bare Trajectory: the given momentum is used (no refresh), like the fixture
    e, st = case["expect"], tr.stat
    assert (st["tree_depth"].cpu().numpy() == np.array(e["tree_depth"])).all()
    assert (st["n_steps"].cpu().numpy() == np.array(e["n_steps"])).all()
    assert (st["numerical_error"].cpu().numpy().astype(bool) == np.array(e["numerical_error"])).all()
    z = tr.z
    for got, want in ((z.theta, e["theta"]), (z.r, e["r"]), (z.lp.gradient, e["lp_gradient"])):
        assert rel_err(got.cpu().numpy(), np.array(want)) < TOL
    assert np.allclose(z.lp.value.cpu().numpy(), e["lp_value"], rtol=1e-10, atol=1e-10)
    assert np.allclose(z.lk.value.cpu().numpy(), e["lk_value"], rtol=1e-10, atol=1e-10)
    assert np.allclose(st["acceptance_rate"].cpu().numpy(), e["acceptance_rate"], rtol=1e-10)
    assert np.allclose(st["hamiltonian_energy_error"].cpu().numpy(), e["hamiltonian_energy_error"], rtol=1e-9, atol=1e-10)
    assert np.allclose(st["max_hamiltonian_energy_error"].cpu().numpy(), e["max_hamiltonian_energy_error"], rtol=1e-9, atol=1e-10)


def test_nuts_max_depth_and_divergence_flags():
    # tiny step size -> every chain hits max_depth (:691); huge step size on the funnel -> divergences (:503-507)
    tr, zo, so = _nuts_case("std_normal", "unit", 4, 64, 0.01, seed=5, max_depth=5)
    assert (F(tr.stat["tree_depth"]) == 5).all() and (so.tree_depth == 5).all()
    assert (F(tr.stat["n_steps"]) == 31).all()
    assert_pp_close(tr.z, zo)
    tr, zo, so = _nuts_case("funnel", "unit", 6, 128, 3.0, seed=6, max_depth=8, scale=3.0)
    assert so.numerical_error.sum() > 0
    assert (F(tr.stat["numerical_error"]) == so.numerical_error).all()
    assert (F(tr.stat["n_steps"]) == so.n_steps).all()
    ok = so.numerical_error == 0
    assert rel_err(F(tr.z.theta)[:, ok], zo.theta[:, ok]) < TOL


def test_nuts_sampling_moments_philox():
    """many-chain NUTS with on-device Philox randomness recovers the target moments (test/sampler.jl style)."""
    D, N = 6, 2048
    m, s = np.linspace(-2, 2, D), np.exp(np.linspace(-1, 1, D))
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.DiagGaussian(m, s))
    zero = lambda: torch.zeros((N, D), dtype=torch.float64, device=DEV)
    z = A.phasepoint(h, zero(), zero())
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.6), A.GeneralisedNoUTurn()))
    rng = A.PhiloxRNG(11)
    depths = []
    for _ in range(40):
        tr = A.transition(rng, h, kern, z)
        z = tr.z
        depths.append(tr.stat["tree_depth"].double().mean().item())
    th = z.theta.cpu().numpy()
    assert np.abs((th.mean(axis=0) - m) / s).max() < 0.12 and np.abs(th.std(axis=0) / s - 1).max() < 0.1
    assert 1.0 < np.mean(depths) < 5.0
    assert tr.stat["acceptance_rate"].mean().item() > 0.6


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("up,down,chunks", [("ce1", "ce", "0"), ("ce3", "ce", "5"), ("ce3", "direct", "0"),
                                            ("direct", "direct", "3"), ("direct", "ce", "2"), (None, None, None)])
def test_pipelined_host_path_equals_device_path(up, down, chunks, pinned, monkeypatch):
    """host-buffer calls with N >= 256 take the chunked upload / kernel / download lane: same bytes out as the device
    call for every transport (copy engines on one or three streams, direct loads / stores on page-locked buffers,
    ragged chunk counts, library defaults), with pageable and with page-locked arrays."""
    if up is not None:
        monkeypatch.setenv("AHMC_PIPE_UP", up)
        monkeypatch.setenv("AHMC_PIPE_DOWN", down)
        monkeypatch.setenv("AHMC_PIPE_CHUNKS", chunks)
    D, N = 100, 4099
    rng = np.random.default_rng(5)
    s = np.exp(rng.uniform(-1, 1, D))
    m = rng.normal(size=D)
    hold = []

    def buf(a):
        if not pinned:
            return np.ascontiguousarray(a)
        t = torch.as_tensor(np.ascontiguousarray(a)).pin_memory()
        hold.append(t)
        return t.numpy()

    Minv_pc = np.exp(rng.uniform(-1, 1, (N, D)))
    th, r = rng.normal(size=(N, D)), rng.normal(size=(N, D))
    eps = 0.05 * np.exp(rng.uniform(-0.3, 0.3, N))
    for Minv in (np.exp(rng.uniform(-1, 1, D)), Minv_pc):
        hd = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s))
        zd, infod = A.step(A.Leapfrog(torch.as_tensor(eps, device=DEV)), hd,
                           A.phasepoint(hd, torch.as_tensor(th, device=DEV), torch.as_tensor(r, device=DEV)), 17, return_info=True)
        hh = A.Hamiltonian(A.DiagEuclideanMetric(buf(Minv)), A.DiagGaussian(m, s))
        z0 = A.phasepoint(hh, buf(th), buf(r))
        z0.lp.gradient = buf(z0.lp.gradient)
        out = None
        if pinned:
            out = A.PhasePoint(buf(np.zeros((N, D))), buf(np.zeros((N, D))), A.DualValue(buf(np.zeros(N)), buf(np.zeros((N, D)))),
                               A.DualValue(buf(np.zeros(N)), buf(np.zeros((N, D)))))
        zh, infoh = A.step(A.Leapfrog(buf(eps)), hh, z0, 17, return_info=True, out=out)
        for a, b in [(zh.theta, zd.theta), (zh.r, zd.r), (zh.lp.value, zd.lp.value), (zh.lk.value, zd.lk.value),
                     (zh.lp.gradient, zd.lp.gradient), (zh.lk.gradient, zd.lk.gradient), (infoh.steps_done, infod.steps_done)]:
            assert np.array_equal(a, b.cpu().numpy())


@pytest.mark.parametrize("model,metric,D,N", [("diag_gauss", "diag", 128, 300), ("diag_gauss", "diag", 100, 300), ("std_normal", "unit", 64, 77),
                                              ("funnel", "diag", 20, 130), ("dense_gauss", "dense", 12, 50), ("diag_gauss", "unit", 7, 19)])
def test_step_without_cached_gradient_equals_step_with_it(model, metric, D, N):
    """z_in.lp_gradient == NULL (a third less upload for host callers): the device recomputes dH/dtheta at the start point,
    so the result is bit-identical to the call that was handed the cached gradient -- fast path (interleaved and
    lane-contiguous layouts), exact path, dense fallback; device and host buffers."""
    rng = np.random.default_rng(40 + D)
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.7, 0.7, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.7, 0.7, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    th, r = rng.normal(size=(D, N)) * (0.3 if model == "funnel" else 1.0), rng.normal(size=(D, N))
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.5))
    z0 = A.phasepoint(h, T(th), T(r))
    zg = A.step(A.Leapfrog(0.07), h, z0, 9)
    zn = A.step(A.Leapfrog(0.07), h, A.PhasePoint(z0.theta, z0.r, A.DualValue(None, None), A.DualValue(None, None)), 9)
    for a, b in [(zg.theta, zn.theta), (zg.r, zn.r), (zg.lp.gradient, zn.lp.gradient), (zg.lp.value, zn.lp.value), (zg.lk.value, zn.lk.value)]:
        if "dense" in (model, metric):  # with the gradient: tiled DMMA kernel; without: warp-per-chain kernel (other summation order)
            assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-13
        else:
            assert torch.equal(a, b)
    thh, rh = np.ascontiguousarray(np.asarray(th).T), np.ascontiguousarray(np.asarray(r).T)
    zh = A.step(A.Leapfrog(0.07), h, A.PhasePoint(thh, rh, A.DualValue(None, None), A.DualValue(None, None)), 9)
    assert np.array_equal(zh.theta, zn.theta.cpu().numpy()) and np.array_equal(zh.lp.gradient, zn.lp.gradient.cpu().numpy())
    with pytest.raises(A.InvalidArgument):  # zero steps hands z back unchanged and needs the gradient to do so
        A.step(A.Leapfrog(0.07), h, A.PhasePoint(z0.theta, z0.r, A.DualValue(None, None), A.DualValue(None, None)), 0)


def test_host_lane_autotune_tries_every_transport_and_stays_bit_identical(monkeypatch):
    """page-locked buffers: the first 12 calls of a shape walk through the four transports (3 rounds), then the fastest is
    kept; every call returns the same bytes as the device call; ahmc_last_transport names what was used."""
    for k in ("AHMC_PIPE_UP", "AHMC_PIPE_DOWN", "AHMC_PIPE_CHUNKS", "AHMC_PIPE_OCC", "AHMC_PIPE_AUTOTUNE"):
        monkeypatch.delenv(k, raising=False)
    D, N = 128, 2051
    m, s, Minv, th, r = synth_diag_gauss(D, N, seed=9)
    h = A.Hamiltonian(A.DiagEuclideanMetric(Minv), A.DiagGaussian(m, s))
    zd = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, T(th), T(r)), 32)
    pin = lambda a: torch.as_tensor(np.ascontiguousarray(a)).pin_memory()
    hold = [pin(th.T), pin(r.T)] + [pin(np.zeros((N, D))) for _ in range(3)] + [pin(np.zeros(N)) for _ in range(2)]
    zin = A.PhasePoint(hold[0].numpy(), hold[1].numpy(), A.DualValue(None, None), A.DualValue(None, None))
    zout = A.PhasePoint(hold[2].numpy(), hold[3].numpy(), A.DualValue(hold[5].numpy(), hold[4].numpy()), A.DualValue(hold[6].numpy(), None))
    plan = A.StepPlan(A.Leapfrog(0.1), h, zin, 32, out=zout)
    ctx = A.get_context(0)
    seen = []
    for i in range(16):
        for t in hold[2:]:
            t.zero_()
        plan()
        seen.append(ctx.last_transport())
        for a, b in [(zout.theta, zd.theta), (zout.r, zd.r), (zout.lp.gradient, zd.lp.gradient), (zout.lp.value, zd.lp.value),
                     (zout.lk.value, zd.lk.value)]:
            assert np.array_equal(a, b.cpu().numpy()), (i, seen[-1])
    assert len(set(seen[:4])) == 4 and all("trial" in t for t in seen[:12])
    assert all("(autotuned)" in t for t in seen[12:]) and len(set(seen[12:])) == 1


def test_small_host_buffer_calls_first_on_a_fresh_context_stay_inside_the_staging_arena():
    """ADVICE r1 (high): the staging arena was sized from grouped reservations while every staged array is rounded up to
    256 B on its own, so N = 1 / small-D host calls made FIRST in a process wrote past the arena.  A fresh interpreter makes
    them first (phasepoint, step, static transition, NUTS) under compute-sanitizer-free conditions by checking results
    against device calls; the arena is now sized from the very arrays a call stages, each rounded up on its own."""
    import subprocess, sys, os
    code = r'''
import numpy as np, torch, ahmc_b200 as A
rng = np.random.default_rng(0)
D, N = 10, 1
h = A.Hamiltonian(A.DiagEuclideanMetric(np.exp(rng.uniform(-1, 1, D))), A.DiagGaussian(rng.normal(size=D), np.exp(rng.uniform(-1, 1, D))))
th, r = rng.normal(size=(N, D)), rng.normal(size=(N, D))
zh = A.phasepoint(h, th, r)                                            # FIRST call of the process: host mode, 7 tiny arrays
zd = A.phasepoint(h, torch.as_tensor(th, device="cuda"), torch.as_tensor(r, device="cuda"))
assert np.array_equal(zh.lp.gradient, zd.lp.gradient.cpu().numpy()) and np.array_equal(zh.lk.value, zd.lk.value.cpu().numpy())
z1h, z1d = A.step(A.Leapfrog(0.1), h, zh, 5), A.step(A.Leapfrog(0.1), h, zd, 5)
assert np.array_equal(z1h.theta, z1d.theta.cpu().numpy()) and np.array_equal(z1h.lk.gradient, z1d.lk.gradient.cpu().numpy())
k = A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.1), A.FixedNSteps(4)))
th_, td_ = A.transition(A.PhiloxRNG(3), h, k, zh), A.transition(A.PhiloxRNG(3), h, k, zd)
assert np.array_equal(th_.z.theta, td_.z.theta.cpu().numpy())
kn = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.2), A.GeneralisedNoUTurn()))
nh, nd = A.transition(A.PhiloxRNG(5), h, kn, zh), A.transition(A.PhiloxRNG(5), h, kn, zd)
assert np.array_equal(nh.z.theta, nd.z.theta.cpu().numpy()) and int(nh.stat["n_steps"][0]) == int(nd.stat["n_steps"][0])
print("ok")
'''
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pr = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=root, timeout=300)
    assert pr.returncode == 0 and "ok" in pr.stdout, pr.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ user closure (split-step)
def _torch_funnel(th):
    """Neal's funnel written by a 'user' in plain torch, gradient by autograd."""
    th = th.detach().clone().requires_grad_(True)
    v, x = th[:, 0], th[:, 1:]
    lp = -v * v / 18 - 0.5 * ((x * x) * torch.exp(-v)[:, None]).sum(dim=1) - 0.5 * (th.shape[1] - 1) * v
    (g,) = torch.autograd.grad(lp.sum(), th)
    return lp.detach(), g


@pytest.mark.parametrize("metric,D", [("unit", 8), ("diag", 40), ("dense", 12)])
def test_callback_target_matches_builtin_and_oracle(metric, D):
    """`Hamiltonian(metric, user_lp, user_grad)`: an arbitrary closure in split-step mode gives the same trajectory."""
    rng = np.random.default_rng(D)
    N = 77
    Minv = None
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    th, r = rng.normal(size=(D, N)) * 0.5, rng.normal(size=(D, N))
    om, ome = oc.Model(oc.FUNNEL, D), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, r)
    zo, st_o, dn_o = oc.leapfrog(om, ome, 0.07, z0o, 9)
    hc = A.Hamiltonian(make_metric(metric, Minv, D), A.CallbackTarget(D, _torch_funnel))
    z0 = A.phasepoint(hc, T(th), T(r))
    assert_pp_close(z0, z0o, tol=1e-12, fields=("lp_gradient", "lp_value", "lk_value", "lk_gradient"))
    z1, info = A.step(A.Leapfrog(0.07), hc, z0, 9, return_info=True)
    assert hc.target.error is None
    assert (F(info.steps_done) == dn_o).all() and (F(info.status) == 0).all()
    assert_pp_close(z1, zo, fields=("theta", "r", "lp_gradient", "lp_value", "lk_value", "lk_gradient"))
    # tempered + backward through the same path
    zo2, _, _ = oc.leapfrog(om, ome, 0.05, z0o, -6, temper_alpha=1.1)
    z2 = A.step(A.TemperedLeapfrog(0.05, 1.1), hc, z0, -6)
    assert_pp_close(z2, zo2)
    # static HMC transition with tapes: same accept decisions and state as the oracle
    nt, et = rng.normal(size=(D, N)), rng.exponential(size=N) * 0.02
    zt, so = oc.hmc_transition(om, ome, 0.12, 7, z0o, nt, et)
    tau = A.Trajectory(A.EndPointTS, A.Leapfrog(0.12), A.FixedNSteps(7))
    tr = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(et, device=DEV)), hc, A.HMCKernel(tau), z0)
    assert (F(tr.stat["is_accept"]).astype(bool) == so.is_accept.astype(bool)).all()
    assert_pp_close(tr.z, zt)
    assert rel_err(F(tr.stat["acceptance_rate"]), so.acceptance_rate) < 1e-9


def test_callback_nonfinite_freeze_and_error_propagation():
    D, N = 3, 5
    def std_normal(th):
        return -0.5 * (th * th).sum(dim=1), -th
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.CallbackTarget(D, std_normal))
    th = np.ones((D, N)); th[:, 1] = 1e200
    om, ome = oc.Model(oc.STD_NORMAL, D), oc.Metric(oc.UNIT)
    z0o = oc.phasepoint(om, ome, th, np.ones((D, N)))
    for compat in (False, True):
        zo, st_o, dn_o = oc.leapfrog(om, ome, 0.1, z0o, 4, compat_break_all=compat)
        z1, info = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, T(th), T(np.ones((D, N)))), 4,
                          flags=A.FLAG_COMPAT_BREAK_ALL if compat else 0, return_info=True)
        assert (F(info.steps_done) == dn_o).all() and (F(info.status) == st_o).all()
        ok = [0, 2, 3, 4]
        assert rel_err(F(z1.theta)[:, ok], zo.theta[:, ok]) < TOL
    def broken(th):
        raise RuntimeError("user model failed")
    hb = A.Hamiltonian(A.UnitEuclideanMetric(D), A.CallbackTarget(D, broken))
    with pytest.raises(A.AhmcError, match="callback"):
        A.phasepoint(hb, T(th), T(th))
    assert isinstance(hb.target.error, RuntimeError)
    with pytest.raises(A.AhmcError, match="NUTS"):
        A.transition(A.PhiloxRNG(0), h, A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.1), A.GeneralisedNoUTurn())),
                     A.phasepoint(h, T(np.ones((D, N))), T(np.ones((D, N)))))


# ------------------------------------------------------------------------------------------------ persistent sampling
@pytest.mark.parametrize("kind", ["hmc", "nuts"])
@pytest.mark.parametrize("D", [5, 128])
def test_multi_transition_launch_equals_sequential_transitions(kind, D):
    """One launch of T transitions (chains free-running) == T single-transition launches with the same Philox
    counters: the persistent loop changes scheduling, not results (sampler.jl:182-228)."""
    N, T = 300, 6
    rng0 = np.random.default_rng(D)
    s = np.exp(rng0.uniform(-0.5, 0.5, D))
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.DiagGaussian(rng0.normal(size=D), s))
    th = torch.as_tensor(rng0.normal(size=(N, D)), device=DEV)
    z0 = A.phasepoint(h, th, torch.zeros_like(th))
    if kind == "hmc":
        kern = A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.5), A.FixedNSteps(7)))
    else:
        kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.35), A.GeneralisedNoUTurn(6, 1000.0)))
    zl, draws, st = A.sample_transitions(A.PhiloxRNG(99), h, kern, z0, T)
    rng = A.PhiloxRNG(99)
    z = z0
    for t in range(T):
        tr = A.transition(rng, h, kern, z)
        z = tr.z
        assert torch.equal(draws[t], z.theta), t
        for k in ("n_steps", "acceptance_rate", "hamiltonian_energy_error", "is_accept", "numerical_error"):
            assert torch.equal(st[k][t], tr.stat[k]), (k, t)
        if kind == "nuts":
            assert torch.equal(st["tree_depth"][t], tr.stat["tree_depth"])
    assert torch.equal(zl.theta, z.theta) and torch.equal(zl.r, z.r) and torch.equal(zl.lp.value, z.lp.value)
    assert torch.equal(zl.lp.gradient, z.lp.gradient) and torch.equal(zl.lk.value, z.lk.value)
    if kind == "nuts":
        assert len(set(st["tree_depth"].flatten().tolist())) > 1


# ------------------------------------------------------------------------------------------------ refreshment / step-size search
def test_partial_momentum_refreshment_vs_oracle():
    """PartialMomentumRefreshment(alpha): r' = alpha r + sqrt(1-alpha^2) xi (hamiltonian.jl:222-254), HMC and NUTS."""
    rng = np.random.default_rng(12)
    D, N, alpha = 9, 150, 0.7
    s = np.exp(rng.uniform(-0.5, 0.5, D))
    m = rng.normal(size=D)
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s), oc.Metric(oc.DIAG, s * s)
    th, r = rng.normal(size=(D, N)), rng.normal(size=(D, N)) / s[:, None]
    z0o = oc.phasepoint(om, ome, th, r)
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.DiagGaussian(m, s, normalised=False))
    z0 = A.phasepoint(h, T(th), T(r))
    nt, et = rng.normal(size=(D, N)), rng.exponential(size=N) * 0.05
    oc.set_partial_refresh(alpha)
    try:
        zo, so = oc.hmc_transition(om, ome, 0.5, 6, z0o, nt, et)
        dirs = rng.integers(0, 2, size=(N, 11)).astype(np.uint8)
        exps = rng.exponential(size=(N, 1024))
        zn, sn, _ = oc.nuts_transition(om, ome, 0.4, z0o, nt, dirs, exps)
    finally:
        oc.set_partial_refresh(0.0)
    ref = A.PartialMomentumRefreshment(alpha)
    tr = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(et, device=DEV)), h,
                      A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.5), A.FixedNSteps(6)), ref), z0)
    assert (F(tr.stat["is_accept"]).astype(bool) == so.is_accept.astype(bool)).all()
    assert_pp_close(tr.z, zo)
    tn = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(exps, device=DEV), dirs=torch.as_tensor(dirs, device=DEV)), h,
                      A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.4), A.GeneralisedNoUTurn()), ref), z0)
    assert (F(tn.stat["n_steps"]) == sn.n_steps).all()
    assert_pp_close(tn.z, zn)
    # with alpha the refreshed momentum stays correlated with the old one
    full = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(et, device=DEV)), h,
                        A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.5), A.FixedNSteps(6))), z0)
    assert not torch.equal(full.z.theta, tr.z.theta)


@pytest.mark.parametrize("model,metric,D", [("diag_gauss", "diag", 128), ("funnel", "unit", 10), ("dense_gauss", "dense", 40),
                                            ("diag_gauss", "dense", 256)])
def test_tempered_leapfrog_inside_transitions_vs_oracle(model, metric, D):
    """`TemperedLeapfrog(eps, alpha)` as the integrator of whole transitions (the reference's sampler matrix runs every
    integrator through every trajectory, test/sampler.jl:81-91): static end point (one n-step `step`, trajectory.jl:337),
    static multinomial (two legs, each tempering by its own n, :374-376) and NUTS (every leaf a 1-step `step`, :640)."""
    rng = np.random.default_rng(900 + D)
    N, alpha = 97, 1.07
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.5, 0.5, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    eps = {"diag_gauss": 0.3, "funnel": 0.15, "dense_gauss": 0.25}[model] * (0.5 if D > 200 else 1.0)
    th = rng.normal(size=(D, N)) * (0.4 if model == "funnel" else 1.0)
    nt, et, ut = rng.normal(size=(D, N)), rng.exponential(size=N) * 0.3, rng.uniform(size=N)
    md = 6
    dirs = rng.integers(0, 2, size=(N, md + 1)).astype(np.uint8)
    exps = rng.exponential(size=(N, 1 << md))
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.0), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, np.zeros((D, N)))
    oc.set_tempering(alpha)
    try:
        zs, ss = oc.hmc_transition(om, ome, eps, 7, z0o, nt, et)
        zm, sm = oc.hmc_multinomial_transition(om, ome, eps, 9, 4, z0o, nt, ut)
        zn, sn, _ = oc.nuts_transition(om, ome, eps, z0o, nt, dirs, exps, max_depth=md)
    finally:
        oc.set_tempering(0.0)
    zu, su, _ = oc.nuts_transition(om, ome, eps, z0o, nt, dirs, exps, max_depth=md)
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.0))
    z0 = A.phasepoint(h, T(th), T(np.zeros((D, N))))
    lf = A.TemperedLeapfrog(eps, alpha)
    ts = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(et, device=DEV)), h,
                      A.HMCKernel(A.Trajectory(A.EndPointTS, lf, A.FixedNSteps(7))), z0)
    assert (F(ts.stat["is_accept"]).astype(bool) == ss.is_accept.astype(bool)).all()
    assert_pp_close(ts.z, zs)
    assert rel_err(F(ts.stat["acceptance_rate"]), ss.acceptance_rate) < 1e-9
    tm = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(ut, device=DEV), n_fwd=4), h,
                      A.HMCKernel(A.Trajectory(A.MultinomialTS, lf, A.FixedNSteps(9))), z0)
    assert (F(tm.stat["tree_depth"]) == sm.tree_depth).all()
    assert_pp_close(tm.z, zm)
    tn = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(exps, device=DEV), dirs=torch.as_tensor(dirs, device=DEV)), h,
                      A.HMCKernel(A.Trajectory(A.MultinomialTS, lf, A.GeneralisedNoUTurn(md, 1000.0))), z0)
    assert (F(tn.stat["n_steps"]) == sn.n_steps).all() and (F(tn.stat["tree_depth"]) == sn.tree_depth).all()
    assert_pp_close(tn.z, zn)
    assert rel_err(F(tn.stat["acceptance_rate"]), sn.acceptance_rate) < 1e-9
    # tempering changes the trees: the untempered transition on the same tapes is a different one
    assert not np.allclose(sn.acceptance_rate, su.acceptance_rate, rtol=1e-6)
    # multi-transition launches accept the tempered integrator and agree with sequential single transitions (Philox)
    if model != "dense_gauss" and metric != "dense":
        k = A.HMCKernel(A.Trajectory(A.EndPointTS, lf, A.FixedNSteps(5)))
        r1, r2 = A.PhiloxRNG(7), A.PhiloxRNG(7)
        zl, draws, _ = A.sample_transitions(r1, h, k, z0, 3)
        zq = z0
        for _ in range(3):
            zq = A.transition(r2, h, k, zq).z
        assert torch.equal(zl.theta, zq.theta)
    with pytest.raises(A.InvalidArgument):
        A.transition(A.PhiloxRNG(1), h, A.HMCKernel(A.Trajectory(A.EndPointTS, A.TemperedLeapfrog(eps, float("nan")), A.FixedNSteps(3))), z0)


def test_find_good_stepsize_batched_equals_per_chain_search():
    """N lock-step copies of the reference's search == the single-chain search run chain by chain on the same momenta;
    host (numpy) positions give the same step sizes as device positions."""
    D, N = 10, 37
    rng = np.random.default_rng(8)
    s = np.exp(rng.uniform(-1.5, 1.5, D))
    h = A.Hamiltonian(A.DiagEuclideanMetric(np.exp(rng.uniform(-0.5, 0.5, D))), A.DiagGaussian(rng.normal(size=D), s))
    th = rng.normal(size=(N, D)) * np.exp(rng.uniform(-2, 2, (N, 1)))  # chains at very different energy scales
    xi = rng.normal(size=(N, D))
    eps_b = A.find_good_stepsize_batched(A.TapeRNG(normal=torch.as_tensor(xi, device=DEV)), h, torch.as_tensor(th, device=DEV))
    eps_1 = [A.find_good_stepsize(A.TapeRNG(normal=torch.as_tensor(xi[c:c + 1], device=DEV)), h, torch.as_tensor(th[c], device=DEV))
             for c in range(N)]
    assert np.array_equal(eps_b.cpu().numpy(), np.array(eps_1))
    eps_h = A.find_good_stepsize_batched(A.TapeRNG(normal=xi), h, th)
    assert np.array_equal(eps_h, np.array(eps_1))


def test_find_good_stepsize_matches_reference_logic():
    """src/trajectory.jl:768-837 restated on the CPU oracle with the same momentum draw -> same eps."""
    D = 12
    rng = np.random.default_rng(3)
    s = np.exp(rng.uniform(-1, 1, D))
    m = rng.normal(size=D)
    h = A.Hamiltonian(A.DiagEuclideanMetric(np.ones(D)), A.DiagGaussian(m, s, normalised=False))
    th = rng.normal(size=D)
    xi = rng.normal(size=(D, 1))
    eps = A.find_good_stepsize(A.TapeRNG(normal=T(xi)), h, torch.as_tensor(th, device=DEV))
    # oracle-side restatement
    om, ome = oc.Model(oc.DIAG_GAUSS, D, m, s), oc.Metric(oc.DIAG, np.ones(D))
    z = oc.phasepoint(om, ome, th[:, None], xi)
    H = z.energy()[0]
    Af = lambda e: oc.leapfrog(om, ome, e, z, 1)[0].energy()[0]
    e = ep = 0.1
    lo, cross, hi = 2 * np.log(0.5), np.log(0.5), np.log(0.75)
    too_high = (H - Af(e)) > cross
    for _ in range(100):
        ep = 2 * e if too_high else 0.5 * e
        if too_high != ((H - Af(e)) > cross):
            break
        e = ep
    e, ep = min(e, ep), max(e, ep)
    for _ in range(100):
        mid = 0.5 * (e + ep)
        dH = H - Af(mid)
        if dH > hi:
            e = mid
        elif dH < lo:
            ep = mid
        else:
            e = mid
            break
    assert eps == pytest.approx(e, rel=1e-12) and 0.01 < eps < 10


# ------------------------------------------------------------------------------------------------ trajectory-sampling forms
def test_full_trajectory_mode_vs_oracle():
    """step(...; full_trajectory=Val(true)) (integrator.jl:229,249-261): every intermediate phase point, forward,
    backward and with a chain that stops early."""
    rng = np.random.default_rng(21)
    D, N, L_ = 7, 45, 9
    s = np.exp(rng.uniform(-0.5, 0.5, D))
    om, ome = oc.Model(oc.FUNNEL, D), oc.Metric(oc.DIAG, s * s)
    th, r = rng.normal(size=(D, N)) * 0.5, rng.normal(size=(D, N))
    th[:, 4] = 1e160  # energies overflow at the first step: that chain returns exactly one point
    z0o = oc.phasepoint(om, ome, th, r)
    h = A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.Funnel(D))
    z0 = A.phasepoint(h, T(th), T(r))
    for n in (L_, -L_):
        traj, done_o = oc.leapfrog_trajectory(om, ome, 0.05, z0o, n)
        zs, done = A.step(A.Leapfrog(0.05), h, z0, n, full_trajectory=True)
        assert (F(done) == done_o).all() and done_o[4] == 1 and len(zs) == L_
        ok = [c for c in range(N) if c != 4]
        for i, z in enumerate(zs):
            assert rel_err(F(z.theta)[:, ok], traj["theta"][:, ok, i]) < TOL
            assert rel_err(F(z.r)[:, ok], traj["r"][:, ok, i]) < TOL
            assert rel_err(F(z.lp.value)[ok], traj["lp_value"][ok, i]) < TOL
            assert rel_err(F(z.lk.gradient)[:, ok], traj["lk_gradient"][:, ok, i]) < TOL
        # the last point of the full trajectory is the ordinary step(n)
        zl = A.step(A.Leapfrog(0.05), h, z0, n)
        assert torch.equal(zs[-1].theta[ok], zl.theta[ok])
    assert A.step(A.Leapfrog(0.05), h, z0, 0, full_trajectory=True)[0] == []


@pytest.mark.parametrize("model,metric,D", [("diag_gauss", "diag", 128), ("std_normal", "unit", 5), ("funnel", "unit", 10)])
@pytest.mark.parametrize("n_fwd", [0, 4, 11])
def test_multinomial_static_transition_vs_oracle(model, metric, D, n_fwd):
    """Trajectory{MultinomialTS}(lf, FixedNSteps(11)) (trajectory.jl:344-390) with tapes: same draw, same statistics."""
    rng = np.random.default_rng(D + n_fwd)
    N, L_ = 211, 11
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.5, 0.5, D))
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    th = rng.normal(size=(D, N)) * (0.4 if model == "funnel" else 1.0)
    nt, ut = rng.normal(size=(D, N)), rng.uniform(size=N)
    eps = {"diag_gauss": 0.45, "std_normal": 0.6, "funnel": 0.15}[model]
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.0), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, np.zeros((D, N)))
    zo, so = oc.hmc_multinomial_transition(om, ome, eps, L_, n_fwd, z0o, nt, ut)
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.0))
    z0 = A.phasepoint(h, T(th), T(np.zeros((D, N))))
    tau = A.Trajectory(A.MultinomialTS, A.Leapfrog(eps), A.FixedNSteps(L_))
    tr = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(ut, device=DEV), n_fwd=n_fwd), h, A.HMCKernel(tau), z0)
    off = F(tr.stat["tree_depth"])
    assert (off == so.tree_depth).all() and off.min() >= -(L_ - n_fwd) and off.max() <= n_fwd
    assert len(set(off.tolist())) > 3  # the draw really ranges over the trajectory
    assert_pp_close(tr.z, zo)
    assert rel_err(F(tr.stat["acceptance_rate"]), so.acceptance_rate) < 1e-9
    assert (F(tr.stat["is_accept"]) == 1).all() and (F(tr.stat["n_steps"]) == L_).all()
    assert np.allclose(F(tr.stat["hamiltonian_energy_error"]), so.hamiltonian_energy_error, rtol=0, atol=1e-9 * D)


def test_multinomial_static_sampling_moments_philox():
    """test/sampler-vec.jl:22-29 analogue: Trajectory{MultinomialTS}(lf, FixedNSteps(10)), many chains."""
    D, N = 5, 4096
    m, s = np.array([1.0, -2.0, 0.5, 0.0, 3.0]), np.array([1.0, 0.5, 2.0, 1.5, 0.7])
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.DiagGaussian(m, s))
    zero = lambda: torch.zeros((N, D), dtype=torch.float64, device=DEV)
    z = A.phasepoint(h, zero(), zero())
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.2), A.FixedNSteps(10)))
    rng = A.PhiloxRNG(77)
    nf = set()
    for _ in range(60):
        tr = A.transition(rng, h, kern, z)
        z = tr.z
        nf.add(tr.stat["n_steps_fwd"])
    th = z.theta.cpu().numpy()
    assert np.abs(th.mean(axis=0) - m).max() < 0.15 and np.abs(th.std(axis=0) - s).max() < 0.15
    assert len(nf) > 5 and tr.stat["acceptance_rate"].mean().item() > 0.8


# ------------------------------------------------------------------------------------------------ K4 tiled DMMA path
@pytest.mark.parametrize("model,metric", [("dense_gauss", "diag"), ("dense_gauss", "dense"), ("diag_gauss", "dense"),
                                          ("std_normal", "dense"), ("dense_gauss", "unit")])
@pytest.mark.parametrize("D,N", [(128, 333), (100, 70), (256, 40), (30, 517), (320, 19)])
def test_dense_tile_kernel_vs_oracle(model, metric, D, N):
    """GEMM-shaped operators run on the tiled fp64-MMA kernel (ahmc_dense.cu): ragged tiles, padded D, per-chain eps,
    backward steps, and one chain that forces its tile back onto the exact path."""
    rng = np.random.default_rng(D * 3 + N)
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.5, 0.5, D))
    elif model == "dense_gauss":
        B = rng.normal(size=(D, D))
        p0, p1 = rng.normal(size=D), B @ B.T / D + np.eye(D)
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    th, r = rng.normal(size=(D, N)), rng.normal(size=(D, N))
    th[3 % D, N // 2] = 1e250  # energy overflow at step 1: that chain freezes, its tile goes to the exact kernel
    eps = 0.03 * np.exp(rng.uniform(-0.3, 0.3, N))
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.3), oc.Metric(METRIC_KINDS[metric], Minv)
    z0o = oc.phasepoint(om, ome, th, r)
    h = A.Hamiltonian(make_metric(metric, Minv, D), make_target(model, D, p0, p1, 0.3))
    z0 = A.phasepoint(h, T(th), T(r))
    for n in (7, -4):
        zo, st_o, dn_o = oc.leapfrog(om, ome, eps, z0o, n)
        z1, info = A.step(A.Leapfrog(torch.as_tensor(eps, device=DEV)), h, z0, n, return_info=True)
        assert (F(info.steps_done) == dn_o).all() and dn_o[N // 2] == 1
        assert (F(info.status) == st_o).all()
        ok = [c for c in range(N) if c != N // 2]
        for f, got in [("theta", z1.theta), ("r", z1.r), ("lp_gradient", z1.lp.gradient), ("lk_gradient", z1.lk.gradient)]:
            assert rel_err(F(got)[:, ok], getattr(zo, f)[:, ok]) < TOL, (f, n)
        assert rel_err(F(z1.lp.value)[ok], zo.lp_value[ok]) < TOL and rel_err(F(z1.lk.value)[ok], zo.lk_value[ok]) < TOL
    # the tile path and the exact path agree to rounding
    ze = A.step(A.Leapfrog(torch.as_tensor(eps, device=DEV)), h, z0, 7, flags=A.FLAG_EXACT_CHECKS)
    z1 = A.step(A.Leapfrog(torch.as_tensor(eps, device=DEV)), h, z0, 7)
    ok = [c for c in range(N) if c != N // 2]
    assert rel_err(F(z1.theta)[:, ok], F(ze.theta)[:, ok]) < 1e-12


# ------------------------------------------------------------------------------------------------ pooled adaptor on the device
@pytest.mark.parametrize("adapt_metric", [True, False], ids=["eps+Minv", "eps-only"])
def test_device_pooled_adaptor_equals_host_adaptors_iteration_by_iteration(adapt_metric):
    """ahmc_adapt_exchange_f64 (K5 -> [all-gather] -> device merge + dual averaging + WelfordVar + Stan windows) fed with the
    same (theta, alpha) per iteration as the host-side pooled adaptors (adaptation.py: the restatement of stepsize.jl:178-210,
    massmatrix.jl:141-157, stan_adaptor.jl:137-159 that tests/test_adaptation.py checks against the oracle): step size after
    every iteration, M^-1 after every window end, reset and finalize! agree to 1e-12."""
    from ahmc_b200 import adaptation as ad

    D, N, n_adapts = 37, 300, 46
    windows = (5, 4, 6)
    rng = np.random.default_rng(8)
    dev_ad = ad.PooledDeviceAdaptor(0, D, N, n_adapts, eps0=0.13, delta=0.8, adapt_metric=adapt_metric, init_buffer=windows[0],
                                    term_buffer=windows[1], window_size=windows[2], n_min=3)
    pc = ad.WelfordVar(D, n_min=3) if adapt_metric else ad.UnitMassMatrix()
    host = ad.StanHMCAdaptor(pc, ad.NesterovDualAveraging(0.8, 0.13), *windows)
    host.initialize(n_adapts)
    assert len(host.window_splits) >= 2
    trace = torch.zeros(n_adapts, dtype=torch.float64, device=DEV)
    scale = np.exp(rng.uniform(-1, 1, D))
    for i in range(1, n_adapts + 1):
        th = torch.as_tensor(rng.normal(size=(N, D)) * scale + 0.3, device=DEV)
        al = torch.as_tensor(np.clip(rng.uniform(0.3, 1.4, N), 0, None), device=DEV)
        dev_ad.exchange(th, al, None, trace, flags=0)
        rec = A.adapt_summary(th, al).cpu().numpy()
        host.adapt(rec)
        if i == n_adapts:
            host.finalize()
        s = dev_ad.state()
        assert s["iteration"] == i
        assert np.allclose(s["merged_record"], rec, rtol=1e-13, atol=0)
        assert abs(s["eps"] - host.eps) <= 1e-12 * host.eps, (i, s["eps"], host.eps)
        assert float(dev_ad.eps[0]) == s["eps"] and float(dev_ad.eps[N - 1]) == s["eps"]
        if adapt_metric:
            assert np.allclose(s["Minv"], host.Minv, rtol=1e-12, atol=0), i
            assert np.array_equal(dev_ad.Minv.cpu().numpy(), s["Minv"])
    assert np.allclose(trace.cpu().numpy()[-1], host.eps, rtol=1e-12)
    dev_ad.destroy()


def test_device_pooled_warmup_runs_without_host_syncs_and_adapts_like_the_host_loop():
    """sample_pooled_device (transition, K5, merge + adaptor update per iteration, all on one stream) against sample() with
    the host-side pooled StanHMCAdaptor on the same Philox streams: same step-size trajectory and final M^-1."""
    from ahmc_b200 import adaptation as ad

    D, N, n_adapts, n_samples = 24, 512, 60, 70
    rng = np.random.default_rng(3)
    s = np.exp(rng.uniform(-1, 1, D))
    h = A.Hamiltonian(A.DiagEuclideanMetric(np.ones(D)), A.DiagGaussian(np.zeros(D), s))
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.2), A.GeneralisedNoUTurn(max_depth=6)))
    th0 = torch.as_tensor(rng.normal(size=(N, D)), device=DEV)
    windows = (10, 8, 6)
    rd = ad.sample_pooled_device(A.PhiloxRNG(5), h, kern, th0, n_samples, n_adapts, eps0=0.2, windows=windows, keep_eps_trace=True)
    host = ad.StanHMCAdaptor(ad.WelfordVar(D), ad.NesterovDualAveraging(0.8, 0.2), *windows)
    rh = ad.sample(A.PhiloxRNG(5), h, kern, th0, n_samples, adaptor=host, n_adapts=n_adapts)
    eps_dev = np.array([st["step_size_after"] for st in rd.stats[:n_adapts]])
    eps_host = np.array([rh.stats[k + 1]["step_size"] for k in range(n_adapts - 1)] + [rh.eps])
    assert np.allclose(eps_dev[:-1], eps_host[:-1], rtol=1e-9) and abs(rd.eps - rh.eps) < 1e-9 * rh.eps
    assert np.allclose(rd.Minv, rh.Minv, rtol=1e-9)
    assert np.allclose(rd.Minv, s * s, rtol=0.35)  # and it learned the target's scales
    assert rd.leapfrog_steps == rh.leapfrog_steps


def test_device_pooled_adaptor_over_nccl_two_ranks():
    """the exchange over a real NCCL communicator created through the C ABI (ahmc_comm_create): 2 ranks, ragged chain counts,
    equal to the host adaptors fed with the rank-ordered merge and bit-identical across ranks (scripts/nccl_exchange_check.py);
    needs two GPUs (skipped on a one-GPU box; the driver's multi-GPU bench runs the same code path in `adapt_exchange`)."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pr = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                         "--master-port", "29517", os.path.join(root, "scripts", "nccl_exchange_check.py")],
                        capture_output=True, text=True, cwd=root, timeout=600)
    assert pr.returncode == 0 and "nccl exchange ok" in pr.stdout, pr.stdout[-1500:] + pr.stderr[-3000:]


# ------------------------------------------------------------------------------------------------ user target (NVRTC, fused)
USER_FUNNEL = r'''
__device__ double ahmc_user_logp_grad(const double* th, double* g, int D, const double* p) {
    const double v = th[0], ev = exp(-v);
    double S = 0.0;
    for (int i = 1; i < D; ++i) { g[i] = -th[i] * ev; S += th[i] * th[i] * ev; }
    g[0] = -v / 9.0 + (S - (D - 1)) * 0.5;
    return -v * v / 18.0 - (S + (D - 1) * v) * 0.5;
}
'''
USER_DIAG = r'''
#define AHMC_USER_COORDWISE
__device__ double ahmc_user_coord(int d, double x, const double* p, double* gd) {   // p = [mean_0, 1/s_0^2, mean_1, ...]
    const double diff = x - p[2 * d], g = diff * p[2 * d + 1];
    *gd = -g;
    return -0.5 * diff * g;
}
'''


@pytest.mark.parametrize("which,D,metric", [("funnel", 20, "diag"), ("funnel", 100, "unit"), ("diag", 128, "diag"), ("diag", 7, "dense")])
def test_user_target_compiled_into_the_kernels_equals_the_builtin_target(which, D, metric):
    """AHMC_MODEL_USER: the user's CUDA device function is compiled (NVRTC) into phasepoint / trajectory / static transition /
    find_good_stepsize kernels; results equal the built-in target's (same arithmetic up to summation order: 1e-12), through
    the exact per-step path, with and without a cached input gradient, on device and on host buffers."""
    rng = np.random.default_rng(60 + D)
    N = 77
    Minv = None
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.5, 0.5, D))
    elif metric == "dense":
        B = rng.normal(size=(D, D))
        Minv = B @ B.T / D + 0.5 * np.eye(D)
    if which == "funnel":
        builtin, user = A.Funnel(D, 0.25), A.UserTarget(D, USER_FUNNEL, c0=0.25)
        th = rng.normal(size=(D, N)) * 0.4
    else:
        m, s = rng.normal(size=D), np.exp(rng.uniform(-0.7, 0.7, D))
        builtin = A.DiagGaussian(m, s, normalised=False)
        builtin.c0 = 0.25
        user = A.UserTarget(D, USER_DIAG, params=np.stack([m, 1.0 / s ** 2], axis=1), c0=0.25)
        th = rng.normal(size=(D, N))
    r = rng.normal(size=(D, N))
    hb, hu = A.Hamiltonian(make_metric(metric, Minv, D), builtin), A.Hamiltonian(make_metric(metric, Minv, D), user)
    zb, zu = A.phasepoint(hb, T(th), T(r)), A.phasepoint(hu, T(th), T(r))
    tol = 1e-12
    for a, b in [(zu.lp.value, zb.lp.value), (zu.lp.gradient, zb.lp.gradient), (zu.lk.value, zb.lk.value)]:
        assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < tol
    z1b = A.step(A.Leapfrog(0.05), hb, zb, 11, flags=A.FLAG_EXACT_CHECKS)
    z1u, info = A.step(A.Leapfrog(0.05), hu, zu, 11, return_info=True)
    assert (F(info.steps_done) == 11).all()
    for a, b in [(z1u.theta, z1b.theta), (z1u.r, z1b.r), (z1u.lp.gradient, z1b.lp.gradient), (z1u.lp.value, z1b.lp.value),
                 (z1u.lk.value, z1b.lk.value)]:
        assert rel_err(a.cpu().numpy(), b.cpu().numpy()) < 1e-11
    z1n = A.step(A.Leapfrog(0.05), hu, A.PhasePoint(zu.theta, zu.r, A.DualValue(None, None), A.DualValue(None, None)), 11)
    assert torch.equal(z1n.theta, z1u.theta) and torch.equal(z1n.lp.gradient, z1u.lp.gradient)
    if metric != "dense":  # host buffers (the pipelined lane takes Unit / Diag metrics)
        zh = A.step(A.Leapfrog(0.05), hu, A.PhasePoint(np.ascontiguousarray(th.T), np.ascontiguousarray(r.T), A.DualValue(None, None),
                                                        A.DualValue(None, None)), 11)
        assert np.array_equal(zh.theta, z1u.theta.cpu().numpy())
    # static transition on identical tapes
    nt, et = T(rng.normal(size=(D, N))), torch.as_tensor(rng.exponential(size=N), device=DEV)
    kern = A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(0.1), A.FixedNSteps(7)))
    tb = A.transition(A.TapeRNG(normal=nt, exp=et), hb, kern, zb, flags=A.FLAG_EXACT_CHECKS)
    tu = A.transition(A.TapeRNG(normal=nt, exp=et), hu, kern, zu)
    assert torch.equal(tu.stat["is_accept"], tb.stat["is_accept"]) and rel_err(tu.z.theta.cpu().numpy(), tb.z.theta.cpu().numpy()) < 1e-11
    # find_good_stepsize in one launch
    eb = A.find_good_stepsize_batched(A.TapeRNG(normal=nt), hb, T(th))
    eu = A.find_good_stepsize_batched(A.TapeRNG(normal=nt), hu, T(th))
    assert torch.equal(eb, eu)


@pytest.mark.parametrize("D,eps,scale,metric", [(20, 0.12, 0.6, "diag"), (100, 0.1, 0.5, "diag"), (3, 0.9, 2.0, "unit")])
def test_nuts_on_a_user_target_matches_the_recursive_oracle_on_tapes(D, eps, scale, metric):
    """NUTS (K3) with the user's funnel compiled into the kernel: same trees, draws and statistics as the recursive oracle
    running the built-in funnel, chain by chain, from shared random tapes."""
    N, max_depth = 150, 10
    rng = np.random.default_rng(D * 13 + 5)
    Minv = np.exp(rng.uniform(-0.5, 0.5, D)) if metric == "diag" else None
    th, nt = rng.normal(size=(D, N)) * scale, rng.normal(size=(D, N))
    dirs = rng.integers(0, 2, size=(N, max_depth + 1)).astype(np.uint8)
    exps = rng.exponential(size=(N, 1 << max_depth))
    om, ome = oc.Model(oc.FUNNEL, D, None, None, 0.0), oc.Metric(METRIC_KINDS[metric], Minv)
    zo, so, used = oc.nuts_transition(om, ome, eps, oc.phasepoint(om, ome, th, np.zeros((D, N))), nt, dirs, exps, max_depth=max_depth)
    h = A.Hamiltonian(make_metric(metric, Minv, D), A.UserTarget(D, USER_FUNNEL))
    z0 = A.phasepoint(h, T(th), T(np.zeros((D, N))))
    tau = A.Trajectory(A.MultinomialTS, A.Leapfrog(eps), A.GeneralisedNoUTurn(max_depth, 1000.0))
    tr = A.transition(A.TapeRNG(normal=T(nt), exp=torch.as_tensor(exps, device=DEV), dirs=torch.as_tensor(dirs, device=DEV)), h,
                      A.HMCKernel(tau), z0)
    st = tr.stat
    assert (F(st["tree_depth"]) == so.tree_depth).all() and (F(st["n_steps"]) == so.n_steps).all()
    assert (F(st["numerical_error"]) == so.numerical_error).all()
    assert_pp_close(tr.z, zo)
    assert rel_err(F(st["acceptance_rate"]), so.acceptance_rate) < 1e-9
    # and a persistent multi-transition Philox run samples v ~ N(0, 9)-ish without errors
    zl, draws, s2 = A.sample_transitions(A.PhiloxRNG(2), h, A.HMCKernel(tau), z0, 5)
    assert torch.isfinite(zl.theta).all()


def test_user_target_compile_errors_come_back_as_messages():
    bad = "__device__ double ahmc_user_logp_grad(const double* th, double* g, int D, const double* p) { return nope; }"
    h = A.Hamiltonian(A.UnitEuclideanMetric(4), A.UserTarget(4, bad))
    with pytest.raises(A.AhmcError) as e:
        A.phasepoint(h, torch.zeros((3, 4), dtype=torch.float64, device=DEV), torch.zeros((3, 4), dtype=torch.float64, device=DEV))
    assert "nope" in str(e.value)
    with pytest.raises(A.InvalidArgument):
        A.UserTarget(4, "int x;").handle(A.get_context(0))


# ------------------------------------------------------------------------------------------------ D > 512 (streaming form)
@pytest.mark.parametrize("model,metric,D,N,n_steps", [("diag_gauss", "diag", 700, 9, 12), ("funnel", "diag", 1500, 5, 9), ("std_normal", "unit", 5000, 3, -6),
                                                        ("diag_gauss", "diag_perchain", 513, 7, 5), ("funnel", "unit", 2049, 4, 1)])
def test_step_and_phasepoint_beyond_512_dimensions_vs_oracle(model, metric, D, N, n_steps):
    """the reference has no bound on D (src/metric.jl:52-72); beyond the register-resident layouts (D <= 512) `step` and
    `phasepoint` stream the chain through registers in tiles of 512 coordinates (ahmc_bigd.cu): same oracle, same tolerance,
    device and host buffers, with and without a cached gradient, per-chain step sizes, backward."""
    rng = np.random.default_rng(D)
    p0 = p1 = Minv = None
    if model == "diag_gauss":
        p0, p1 = rng.normal(size=D), np.exp(rng.uniform(-0.7, 0.7, D))
    mk = "diag" if metric == "diag_perchain" else metric
    if metric == "diag":
        Minv = np.exp(rng.uniform(-0.7, 0.7, D))
    elif metric == "diag_perchain":
        Minv = np.exp(rng.uniform(-0.7, 0.7, (D, N)))
    th, r = rng.normal(size=(D, N)) * (0.05 if model == "funnel" else 1.0), rng.normal(size=(D, N))
    eps = 0.02 * np.exp(rng.uniform(-0.3, 0.3, N))
    om, ome = oc.Model(MODEL_KINDS[model], D, p0, p1, 0.5), oc.Metric(METRIC_KINDS[mk], Minv)
    z0o = oc.phasepoint(om, ome, th, r)
    zo, st_o, dn_o = oc.leapfrog(om, ome, eps, z0o, n_steps)
    h = A.Hamiltonian(make_metric(mk, Minv, D), make_target(model, D, p0, p1, 0.5))
    z0 = A.phasepoint(h, T(th), T(r))
    assert_pp_close(z0, z0o, tol=1e-12, fields=("lp_gradient", "lp_value", "lk_value", "lk_gradient"))
    lf = A.Leapfrog(torch.as_tensor(eps, device=DEV))
    z1, info = A.step(lf, h, z0, n_steps, return_info=True)
    assert (F(info.steps_done) == dn_o).all()
    assert_pp_close(z1, zo, fields=("theta", "r", "lp_gradient", "lp_value", "lk_value", "lk_gradient"))
    zn = A.step(lf, h, A.PhasePoint(z0.theta, z0.r, A.DualValue(None, None), A.DualValue(None, None)), n_steps)
    assert torch.equal(zn.theta, z1.theta) and torch.equal(zn.lp.gradient, z1.lp.gradient)
    zi = A.PhasePoint(z0.theta.clone(), z0.r.clone(), A.DualValue(z0.lp.value.clone(), z0.lp.gradient.clone()), A.DualValue(z0.lk.value.clone(), None))
    zi2 = A.step(lf, h, zi, n_steps, out=zi)  # in place
    assert torch.equal(zi2.theta, z1.theta) and torch.equal(zi2.r, z1.r)
    if metric != "diag_perchain":
        zh = A.step(A.Leapfrog(eps), h, A.PhasePoint(np.ascontiguousarray(th.T), np.ascontiguousarray(r.T), A.DualValue(None, None),
                                                      A.DualValue(None, None)), n_steps)
        assert np.array_equal(zh.theta, z1.theta.cpu().numpy()) and np.array_equal(zh.lk.value, z1.lk.value.cpu().numpy())


def test_beyond_512_dimensions_nonfinite_freeze_and_unsupported_combinations():
    D, N = 600, 4
    h = A.Hamiltonian(A.UnitEuclideanMetric(D), A.StdNormal(D))
    th = np.ones((N, D))
    th[2, 77] = 1e200
    z1, info = A.step(A.Leapfrog(0.1), h, A.phasepoint(h, torch.as_tensor(th, device=DEV), torch.ones((N, D), dtype=torch.float64, device=DEV)), 5,
                      return_info=True)
    assert list(F(info.steps_done)) == [5, 5, 1, 5] and list(F(info.status)) == [0, 0, 1, 0] and float(z1.lp.value[2]) == -np.inf
    hd = A.Hamiltonian(A.DenseEuclideanMetric(np.eye(D)), A.StdNormal(D))
    with pytest.raises(A.AhmcError):
        A.phasepoint(hd, torch.zeros((N, D), dtype=torch.float64, device=DEV), torch.zeros((N, D), dtype=torch.float64, device=DEV))
    kern = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(0.1), A.GeneralisedNoUTurn()))
    with pytest.raises(A.AhmcError):
        A.transition(A.PhiloxRNG(1), h, kern, A.phasepoint(h, torch.zeros((N, D), dtype=torch.float64, device=DEV), torch.zeros((N, D), dtype=torch.float64, device=DEV)))
