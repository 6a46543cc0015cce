"""Host-buffer staging (AHMC_FLAG_HOST_BUFFERS): every entry point called on numpy arrays stages them through the
context's device arena and must return, bit for bit, what the same call returns on CUDA tensors -- every output array,
every stats field, status and steps_done.  Ragged N; D = 40, where both the tiled K4 trajectory and the cooperative NUTS
form run; per-chain step sizes and per-chain M^-1 wherever the entry point takes them."""
import numpy as np
import pytest
import torch

import ahmc_b200 as A

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
D, N = 40, 37


def dev(x):
    return torch.as_tensor(x, device=DEV)


def same(got_h, got_d, what):
    a = np.asarray(got_h)
    b = got_d.cpu().numpy() if isinstance(got_d, torch.Tensor) else np.asarray(got_d)
    if a.dtype == np.uint32 and b.dtype == np.int32:  # torch holds the uint32 status words as int32
        b = b.view(np.uint32)
    assert a.dtype == b.dtype and a.shape == b.shape, (what, a.dtype, b.dtype, a.shape, b.shape)
    assert np.array_equal(a, b, equal_nan=True), what


def same_pp(zh, zd, what):
    same(zh.theta, zd.theta, what + ".theta")
    same(zh.r, zd.r, what + ".r")
    same(zh.lp.value, zd.lp.value, what + ".lp.value")
    same(zh.lp.gradient, zd.lp.gradient, what + ".lp.gradient")
    same(zh.lk.value, zd.lk.value, what + ".lk.value")
    assert (zh.lk.gradient is None) == (zd.lk.gradient is None), what
    if zh.lk.gradient is not None:
        same(zh.lk.gradient, zd.lk.gradient, what + ".lk.gradient")


def same_stats(sh, sd, what, unwritten=()):
    assert sorted(sh) == sorted(sd), what
    for k in sh:
        if k not in unwritten:
            same(sh[k], sd[k], f"{what}.stat[{k}]")


@pytest.fixture(scope="module")
def P():
    rng = np.random.default_rng(20261017)
    mu = rng.normal(size=D)
    s = np.exp(rng.uniform(-0.5, 0.5, D))
    B = rng.normal(size=(D, D))
    Minv_dense = B @ B.T / D + 0.5 * np.eye(D)
    C = rng.normal(size=(D, D))
    prec = C @ C.T / D + 0.5 * np.eye(D)
    p = dict(
        th=rng.normal(size=(N, D)),
        r=rng.normal(size=(N, D)),
        eps=0.12 * np.exp(rng.uniform(-0.2, 0.2, N)),
        normal=rng.normal(size=(N, D)),
        exp1=rng.exponential(size=N),
        unif1=rng.uniform(size=N),
        h_diag=A.Hamiltonian(A.DiagEuclideanMetric(np.exp(rng.uniform(-0.3, 0.3, (N, D)))), A.DiagGaussian(mu, s)),
        h_dense=A.Hamiltonian(A.DenseEuclideanMetric(Minv_dense), A.DenseGaussian(mu, prec)),
        h_cb=A.Hamiltonian(A.DiagEuclideanMetric(s * s), A.CallbackTarget(D, lambda th: (-0.5 * (th * th).sum(dim=1), -th))),
    )
    p["dirs"] = rng.integers(0, 2, size=(N, 7)).astype(np.uint8)
    p["exps"] = rng.exponential(size=(N, 64))
    return p


def pair(h, P):
    """the same starting phase point, once on host arrays and once on device tensors"""
    return A.phasepoint(h, P["th"], P["r"]), A.phasepoint(h, dev(P["th"]), dev(P["r"]))


@pytest.mark.parametrize("ham", ["h_diag", "h_dense", "h_cb"])
def test_phasepoint_and_step(P, ham):
    h = P[ham]
    zh, zd = pair(h, P)
    same_pp(zh, zd, "phasepoint")
    for lf in (A.Leapfrog(P["eps"]), A.Leapfrog(0.1)):
        for n in (5, -3):
            (oh, ih), (od, idd) = (A.step(lf, h, z, n, return_info=True) for z in (zh, zd))
            same_pp(oh, od, f"step({n})")
            same(ih.status, idd.status, "status")
            same(ih.steps_done, idd.steps_done, "steps_done")
    oh, od = (A.step(A.Leapfrog(P["eps"]), h, z, 4, with_lk_gradient=False) for z in (zh, zd))
    same_pp(oh, od, "step without lk_gradient")


def test_compat_break_all_reruns_from_staged_inputs(P):
    h = P["h_diag"]
    zh, zd = pair(h, P)
    eps = P["eps"].copy()
    eps[3] = 1e100  # chain 3 overflows at its first step: every chain stops there and is re-run from the inputs
    (oh, ih), (od, idd) = (A.step(A.Leapfrog(eps), h, z, 6, flags=A.FLAG_COMPAT_BREAK_ALL, return_info=True) for z in (zh, zd))
    assert int(ih.steps_done.max()) < 6
    same_pp(oh, od, "compat step")
    same(ih.status, idd.status, "status")
    same(ih.steps_done, idd.steps_done, "steps_done")


def test_full_trajectory(P):
    h = P["h_diag"]
    zh, zd = pair(h, P)
    (th_, dh), (td_, dd) = (A.step(A.Leapfrog(P["eps"]), h, z, 4, full_trajectory=True) for z in (zh, zd))
    same(dh, dd, "steps_done")
    assert len(th_) == len(td_) == 4
    for i, (a, b) in enumerate(zip(th_, td_)):
        same_pp(a, b, f"trajectory[{i}]")


@pytest.mark.parametrize("ham", ["h_diag", "h_dense"])
def test_rand_momentum(P, ham):
    m = P[ham].metric
    same(A.rand_momentum(A.PhiloxRNG(3), m, None, P["th"]), A.rand_momentum(A.PhiloxRNG(3), m, None, dev(P["th"])), "philox")
    same(A.rand_momentum(A.TapeRNG(normal=P["normal"]), m, None, P["th"]),
         A.rand_momentum(A.TapeRNG(normal=dev(P["normal"])), m, None, dev(P["th"])), "tape")


@pytest.mark.parametrize("ham,sampler", [("h_diag", "endpoint"), ("h_dense", "endpoint"), ("h_cb", "endpoint"),
                                         ("h_diag", "multinomial"), ("h_dense", "multinomial")])
def test_static_transitions(P, ham, sampler):
    """EndPointTS on the dense Hamiltonian runs the unfused K4 transition, on the callback target the split-step one"""
    h = P[ham]
    zh, zd = pair(h, P)
    ts = A.EndPointTS if sampler == "endpoint" else A.MultinomialTS
    exp = P["exp1"] if sampler == "endpoint" else P["unif1"]
    # the static MultinomialTS transition leaves this NUTS field of its stats buffers unwritten
    unwritten = () if sampler == "endpoint" else ("max_hamiltonian_energy_error",)
    k = A.HMCKernel(A.Trajectory(ts, A.Leapfrog(P["eps"]), A.FixedNSteps(6)))
    th_, td_ = A.transition(A.PhiloxRNG(5), h, k, zh), A.transition(A.PhiloxRNG(5), h, k, zd)
    same_pp(th_.z, td_.z, "philox transition")
    same_stats(th_.stat, td_.stat, "philox transition", unwritten)
    th_ = A.transition(A.TapeRNG(normal=P["normal"], exp=exp, n_fwd=2), h, k, zh)
    td_ = A.transition(A.TapeRNG(normal=dev(P["normal"]), exp=dev(exp), n_fwd=2), h, k, zd)
    same_pp(th_.z, td_.z, "tape transition")
    same_stats(th_.stat, td_.stat, "tape transition", unwritten)
    kt = A.Trajectory(ts, A.Leapfrog(0.1), A.FixedNSteps(3))  # a bare trajectory keeps z.r (no refresh)
    th_, td_ = A.transition(A.TapeRNG(exp=exp, n_fwd=1), h, kt, zh), A.transition(A.TapeRNG(exp=dev(exp), n_fwd=1), h, kt, zd)
    same_pp(th_.z, td_.z, "no-refresh transition")
    same_stats(th_.stat, td_.stat, "no-refresh transition", unwritten)


@pytest.mark.parametrize("ham", ["h_diag", "h_dense"])
def test_nuts_transitions(P, ham):
    """the dense Hamiltonian runs the cooperative NUTS form on the staged Minv / cholU; tapes stage the direction and
    exponential draws"""
    h = P[ham]
    zh, zd = pair(h, P)
    k = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(P["eps"]), A.GeneralisedNoUTurn(6, 1000.0)))
    th_, td_ = A.transition(A.PhiloxRNG(7), h, k, zh), A.transition(A.PhiloxRNG(7), h, k, zd)
    same_pp(th_.z, td_.z, "philox nuts")
    same_stats(th_.stat, td_.stat, "philox nuts")
    th_ = A.transition(A.TapeRNG(normal=P["normal"], exp=P["exps"], dirs=P["dirs"]), h, k, zh)
    td_ = A.transition(A.TapeRNG(normal=dev(P["normal"]), exp=dev(P["exps"]), dirs=dev(P["dirs"])), h, k, zd)
    same_pp(th_.z, td_.z, "tape nuts")
    same_stats(th_.stat, td_.stat, "tape nuts")


@pytest.mark.parametrize("kind", ["hmc", "nuts"])
@pytest.mark.parametrize("ham", ["h_diag", "h_dense"])
def test_multi_transition_sampling_with_draws_and_stats(P, kind, ham):
    h = P[ham]
    zh, zd = pair(h, P)
    if kind == "hmc":
        k = A.HMCKernel(A.Trajectory(A.EndPointTS, A.Leapfrog(P["eps"]), A.FixedNSteps(5)))
    else:
        k = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(P["eps"]), A.GeneralisedNoUTurn(5, 1000.0)))
    zlh, dh, sh = A.sample_transitions(A.PhiloxRNG(11), h, k, zh, 4)
    zld, dd, sd = A.sample_transitions(A.PhiloxRNG(11), h, k, zd, 4)
    same_pp(zlh, zld, "last")
    same(dh, dd, "draws")
    same_stats(sh, sd, "sample")


def test_find_good_stepsize_batched(P):
    h = P["h_diag"]
    eh, rh = A.find_good_stepsize_batched(A.PhiloxRNG(13), h, P["th"], return_momentum=True)
    ed, rd = A.find_good_stepsize_batched(A.PhiloxRNG(13), h, dev(P["th"]), return_momentum=True)
    same(eh, ed, "eps")
    same(rh, rd, "momentum")


def test_nuts_adapt_sample(P):
    h = P["h_diag"]
    zh, zd = pair(h, P)
    k = A.HMCKernel(A.Trajectory(A.MultinomialTS, A.Leapfrog(P["eps"]), A.GeneralisedNoUTurn(5, 1000.0)))
    ad = A.VectorisedStanAdaptor(init_buffer=2, term_buffer=2, window_size=2)
    outs_h = A.nuts_adapt_sample(A.PhiloxRNG(17), h, k, zh, 10, 7, ad, keep_eps_trace=True)
    outs_d = A.nuts_adapt_sample(A.PhiloxRNG(17), h, k, zd, 10, 7, ad, keep_eps_trace=True)
    same_pp(outs_h[0], outs_d[0], "last")
    same(outs_h[1], outs_d[1], "draws")
    same_stats(outs_h[2], outs_d[2], "adapt")
    for name, a, b in zip(("eps", "Minv", "eps_trace"), outs_h[3:], outs_d[3:]):
        same(a, b, name)


def test_adapt_summary_and_cov(P):
    alpha = np.random.default_rng(1).uniform(size=N)
    sh, sd = A.adapt_summary(P["th"], alpha), A.adapt_summary(dev(P["th"]), dev(alpha))
    same(sh, sd, "summary")
    mean = sh[2:2 + D].copy()
    same(A.adapt_cov(P["th"], mean), A.adapt_cov(dev(P["th"]), dev(mean)), "cov")
