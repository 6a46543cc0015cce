"""adaptation.py -- host-side mirror of src/adaptation/*.jl for MANY chains with POOLED statistics, and the
`sample` loop (src/sampler.jl:159-248) on top of the fused transition kernels.

The reference adapts per chain and never pools (`src/adaptation/Adaptation.jl:52`: "TODO: implement consensus
adaptor"); many-chain HMCDA / NUTS with one shared step size and metric needs the pooled form (SURVEY.md 8a Q6,
8e).  Each GPU reduces its chains to a (2+2D)-double record with ahmc_adapt_summary_f64 (K5); the records of all
ranks are exchanged with ONE all-gather (torch.distributed / NCCL) and merged in rank order, so every rank computes
bit-identical eps and M^-1.  With one chain on one rank every formula below reduces to the reference's scalar path
(checked against the oracle in tests/test_adaptation.py).  Scalar arithmetic only: this is control logic, not the
hot path.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np

from . import core as A


# ------------------------------------------------------------------------------------------------ records
def merge_records(records: List[np.ndarray], kind: str = "diag") -> np.ndarray:
    """Chan merge of per-rank records in list (= rank) order.  Layouts (D inferred from the size):
       "diag"   [n, sum_alpha, mean[D], M2[D]]
       "nutpie" [n, sum_alpha, mean[D], M2[D], mean_g[D], M2_g[D]]            (positions and gradients)
       "cov"    [n, sum_alpha, mean[D], M2[D], M2full[D*D]]                    (dense second moment)"""
    out = np.array(records[0], dtype=np.float64, copy=True)
    if kind == "diag":
        D = (out.size - 2) // 2
    elif kind == "nutpie":
        D = (out.size - 2) // 4
    elif kind == "cov":
        D = int(round(-1 + math.sqrt(1 + (out.size - 2)))) if out.size > 2 else 0  # D^2 + 2D = size - 2
        assert 2 + 2 * D + D * D == out.size, "bad cov record size"
    else:
        raise ValueError(kind)
    for rec in records[1:]:
        n_a, n_b = out[0], rec[0]
        n = n_a + n_b
        w = n_a * n_b / n
        delta = rec[2:2 + D] - out[2:2 + D]
        out[2 + D:2 + 2 * D] += rec[2 + D:2 + 2 * D] + delta * delta * w
        if kind == "cov":
            out[2 + 2 * D:] += rec[2 + 2 * D:] + (np.outer(delta, delta) * w).ravel()
        out[2:2 + D] += delta * (n_b / n)
        if kind == "nutpie":
            dg = rec[2 + 2 * D:2 + 3 * D] - out[2 + 2 * D:2 + 3 * D]
            out[2 + 3 * D:] += rec[2 + 3 * D:] + dg * dg * w
            out[2 + 2 * D:2 + 3 * D] += dg * (n_b / n)
        out[1] = out[1] + rec[1]
        out[0] = n
    return out


def allgather_records(rec) -> List[np.ndarray]:
    """One all-gather of the tiny adaptor record across ranks (the path's only exchange, SURVEY 8e)."""
    try:
        import torch
        import torch.distributed as dist
    except Exception:  # pragma: no cover
        dist = None
    if dist is None or not dist.is_available() or not dist.is_initialized() or dist.get_world_size() == 1:
        r = rec.detach().cpu().numpy() if hasattr(rec, "detach") else np.asarray(rec)
        return [np.array(r, dtype=np.float64)]
    t = rec if hasattr(rec, "detach") else torch.as_tensor(rec)
    if dist.get_backend() == "nccl" and not t.is_cuda:
        t = t.cuda()
    if dist.get_backend() == "gloo" and t.is_cuda:
        t = t.cpu()
    outs = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(outs, t.contiguous())
    return [o.cpu().numpy().astype(np.float64) for o in outs]


# ------------------------------------------------------------------------------------------------ step size
class NesterovDualAveraging:
    """src/adaptation/stepsize.jl:111-229 with a scalar (shared) step size; `adapt` takes the pooled mean of
    min(1, alpha) over all chains (one chain: exactly stepsize.jl:178-210)."""

    def __init__(self, delta: float, eps: float, gamma: float = 0.05, t_0: float = 10.0, kappa: float = 0.75):
        self.gamma, self.t_0, self.kappa, self.delta = gamma, t_0, kappa, delta
        self.eps = float(eps)
        self.reset()

    def reset(self):  # stepsize.jl:38-44
        self.m, self.mu, self.x_bar, self.H_bar = 0, math.log(10 * self.eps), 0.0, 0.0

    def adapt(self, mean_min1_alpha: float):
        m = self.m + 1
        eta_H = 1.0 / (m + self.t_0)
        H_bar = (1.0 - eta_H) * self.H_bar + eta_H * (self.delta - mean_min1_alpha)
        x = self.mu - H_bar * (math.sqrt(m) / self.gamma)
        eta_x = m ** (-self.kappa)
        x_bar = (1.0 - eta_x) * self.x_bar + eta_x * x
        try:
            eps = math.exp(x)
        except OverflowError:
            eps = math.inf
        if not math.isfinite(eps):  # stepsize.jl:199-203: keep the previous state
            return
        self.m, self.eps, self.x_bar, self.H_bar = m, eps, x_bar, H_bar

    def finalize(self):  # stepsize.jl:54-57
        self.eps = math.exp(self.x_bar)


class FixedStepSize:
    def __init__(self, eps):
        self.eps = eps

    def adapt(self, a): ...
    def reset(self): ...
    def finalize(self): ...


# ------------------------------------------------------------------------------------------------ mass matrix
class WelfordVar:
    """Pooled WelfordVar (src/adaptation/massmatrix.jl:86-157): every chain of every rank contributes one sample
    per iteration; batches arrive as (n, mean, M2) records and are Chan-merged."""

    def __init__(self, D: int, n_min: int = 10):
        self.D, self.n_min = D, n_min
        self.var = np.ones(D)
        self.reset()

    def reset(self):
        self.n, self.mu, self.M = 0.0, np.zeros(self.D), np.zeros(self.D)

    def push_record(self, rec: np.ndarray):
        D = self.D
        n_b, mean_b, M2_b = rec[0], rec[2:2 + D], rec[2 + D:2 + 2 * D]
        n = self.n + n_b
        delta = mean_b - self.mu
        self.M = self.M + M2_b + delta * delta * (self.n * n_b / n)
        self.mu = self.mu + delta * (n_b / n)
        self.n = n

    def get_estimation(self):  # massmatrix.jl:152-157
        n = self.n
        return n / ((n + 5) * (n - 1)) * self.M + 1e-3 * (5 / (n + 5))

    def update(self):  # massmatrix.jl:60-62
        if self.n >= self.n_min:
            self.var = self.get_estimation()


class NutpieVar:
    """Pooled NutpieVar (src/adaptation/massmatrix.jl:172-250): WelfordVar of the positions and of the gradients,
    estimate sqrt(var_theta / var_grad) from the two regularised Welford estimates."""
    record_kind = "nutpie"

    def __init__(self, D: int, n_min: int = 10):
        self.D, self.n_min = D, n_min
        self.pos, self.grad = WelfordVar(D, n_min), WelfordVar(D, n_min)
        self.var = np.ones(D)
        self.n = 0.0

    def reset(self):
        self.n = 0.0
        self.pos.reset()
        self.grad.reset()

    def push_record(self, rec: np.ndarray):
        D = self.D
        self.pos.push_record(rec[:2 + 2 * D])
        self.grad.push_record(np.concatenate([rec[:2], rec[2 + 2 * D:2 + 4 * D]]))
        self.n = self.pos.n

    def get_estimation(self):  # massmatrix.jl:244-248
        return np.sqrt(self.pos.get_estimation() / self.grad.get_estimation())

    def update(self):
        if self.n >= self.n_min:
            self.var = self.get_estimation()


class WelfordCov:
    """Pooled WelfordCov (src/adaptation/massmatrix.jl:286-340): (n, mean, M2 full) records, Chan-merged;
    estimate n/((n+5)(n-1)) M + 1e-3 * 5/(n+5) I.  `var` holds the D x D covariance (-> DenseEuclideanMetric)."""
    record_kind = "cov"

    def __init__(self, D: int, n_min: int = 10):
        self.D, self.n_min = D, n_min
        self.var = np.eye(D)
        self.reset()

    def reset(self):
        self.n, self.mu, self.M = 0.0, np.zeros(self.D), np.zeros((self.D, self.D))

    def push_record(self, rec: np.ndarray):
        D = self.D
        n_b, mean_b, M2_b = rec[0], rec[2:2 + D], rec[2 + 2 * D:2 + 2 * D + D * D].reshape(D, D)
        n = self.n + n_b
        delta = mean_b - self.mu
        self.M = self.M + M2_b + np.outer(delta, delta) * (self.n * n_b / n)
        self.mu = self.mu + delta * (n_b / n)
        self.n = n

    def get_estimation(self):  # massmatrix.jl:335-340
        n = self.n
        return n / ((n + 5) * (n - 1)) * self.M + 1e-3 * (5 / (n + 5)) * np.eye(self.D)

    def update(self):
        if self.n >= self.n_min:
            self.var = self.get_estimation()


def iteration_record(z, acceptance_rate, kind: str = "diag"):
    """This rank's adaptor record of one iteration, built on the device (K5 / K5b), ready for the all-gather."""
    rec = A.adapt_summary(z.theta, acceptance_rate)
    if kind == "diag":
        return rec
    D = z.theta.shape[1]
    if kind == "nutpie":
        extra = A.adapt_summary(z.lp.gradient, None)[2:]
    else:
        extra = A.adapt_cov(z.theta, rec[2:2 + D]).reshape(-1)
    if hasattr(rec, "detach"):
        import torch

        return torch.cat([rec, extra])
    return np.concatenate([rec, extra])


class UnitMassMatrix:
    var = None

    def reset(self): ...
    def push_record(self, rec): ...
    def update(self): ...


# ------------------------------------------------------------------------------------------------ Stan windows
def stan_windows(n_adapts: int, init_buffer: int = 75, term_buffer: int = 50, window_size: int = 25):
    """src/adaptation/stan_adaptor.jl:13-50 -> (window_start, window_end, window_splits)."""
    window_start, window_end = init_buffer + 1, n_adapts - term_buffer
    splits, next_window = [], init_buffer + window_size
    while next_window <= window_end:
        if next_window + 2 * window_size > window_end:
            next_window = window_end
        splits.append(next_window)
        window_size *= 2
        next_window += window_size
    if splits and splits[-1] == n_adapts:
        splits.pop()
    return window_start, window_end, splits


class StanHMCAdaptor:
    """src/adaptation/stan_adaptor.jl:61-159 (3-phase windowed adaptation) on pooled records."""

    def __init__(self, pc, ssa, init_buffer: int = 75, term_buffer: int = 50, window_size: int = 25):
        self.pc, self.ssa = pc, ssa
        self.init_buffer, self.term_buffer, self.window_size = init_buffer, term_buffer, window_size
        self.i, self.window_start, self.window_end, self.window_splits = 0, 0, 0, []

    def initialize(self, n_adapts: int):
        self.window_start, self.window_end, self.window_splits = stan_windows(
            n_adapts, self.init_buffer, self.term_buffer, self.window_size)

    def adapt(self, rec: np.ndarray):
        """rec = merged record of this iteration (stan_adaptor.jl:137-159)."""
        self.i += 1
        self.ssa.adapt(rec[1] / rec[0])
        if self.window_start <= self.i <= self.window_end:
            self.pc.push_record(rec)
            if self.i in self.window_splits:
                self.pc.update()
        if self.i in self.window_splits:
            self.ssa.reset()
            self.pc.reset()

    def finalize(self):
        self.ssa.finalize()

    @property
    def eps(self):
        return self.ssa.eps

    @property
    def Minv(self):
        return self.pc.var


class NaiveHMCAdaptor(StanHMCAdaptor):
    """src/adaptation/Adaptation.jl:41-64: adapt both every iteration, no windows."""

    def initialize(self, n_adapts: int): ...

    def adapt(self, rec: np.ndarray):
        self.i += 1
        self.ssa.adapt(rec[1] / rec[0])
        self.pc.push_record(rec)
        self.pc.update()


# ------------------------------------------------------------------------------------------------ sample
@dataclass
class SampleResult:
    theta: object          # final positions (N, D)
    draws: list            # kept draws (list of (N, D) tensors) if keep_draws
    stats: list            # per-iteration dicts of pooled scalars
    eps: float
    Minv: Optional[np.ndarray]
    leapfrog_steps: int = 0
    timing: dict = field(default_factory=dict)  # wall seconds: transition / adapt / sampling_launch / bookkeeping


def _mean(x):
    return x.double().mean() if hasattr(x, "double") else np.asarray(x, dtype=np.float64).mean()


def _sum(x):
    return x.sum() if hasattr(x, "detach") else np.asarray(x).sum()


def sample(rng, h: A.Hamiltonian, kappa: A.HMCKernel, theta, n_samples: int, adaptor=None, n_adapts: int = 0,
           keep_draws: bool = False, drop_warmup: bool = False, fused_sampling: bool = True) -> SampleResult:
    """`sample(rng, h, kappa, theta, n_samples, adaptor, n_adapts)` (src/sampler.jl:159-248) for N chains on this
    rank, pooled adaptation across chains and ranks.
    Warm-up iterations (i <= n_adapts): one fused transition kernel (K2 / K3), one K5 launch and one all-gather of
    the (2+2D)-double record each -- the adaptor must see iteration i before iteration i+1 starts.
    Sampling iterations (i > n_adapts) have no such dependency: with a Philox RNG they run as ONE persistent launch
    (`sample_transitions`), every chain advancing at its own pace (`fused_sampling=False` keeps the loop)."""
    import time

    import torch

    tm = dict(transition=0.0, adapt=0.0, sampling_launch=0.0, bookkeeping=0.0)
    z = A.phasepoint(h, theta, torch.zeros_like(theta))  # sample_init (sampler.jl:36-46); r is refreshed anyway
    if isinstance(adaptor, A.VectorisedStanAdaptor):
        # the reference's vectorised adaptors (per-chain eps and M^-1): warm-up and sampling are ONE launch
        if not isinstance(h.metric, A.DiagEuclideanMetric):
            raise A.L.AhmcError(A.L.ERR_UNSUPPORTED, "VectorisedStanAdaptor adapts a per-chain diagonal M^-1: DiagEuclideanMetric")
        n_adapts = min(n_adapts, n_samples)
        t0 = time.perf_counter()
        zl, dr, st, eps, minv, trace = A.nuts_adapt_sample(rng, h, kappa, z, n_samples, n_adapts, adaptor,
                                                           keep_draws=keep_draws, keep_eps_trace=True)
        if hasattr(zl.theta, "is_cuda") and zl.theta.is_cuda:
            torch.cuda.synchronize(zl.theta.device)
        tm["sampling_launch"] = time.perf_counter() - t0
        a, e, n = st["acceptance_rate"], st["numerical_error"], st["n_steps"]
        acc_h = (a.double().mean(dim=1).cpu().numpy() if hasattr(a, "detach") else np.asarray(a).mean(axis=1))
        nerr_h = (e.sum(dim=1).cpu().numpy() if hasattr(e, "detach") else np.asarray(e).sum(axis=1))
        nst_h = (n.sum(dim=1).cpu().numpy() if hasattr(n, "detach") else np.asarray(n).sum(axis=1))
        eps_h = (trace.double().mean(dim=1).cpu().numpy() if hasattr(trace, "detach") else np.asarray(trace).mean(axis=1))
        stats = [dict(acceptance_rate=float(acc_h[k]), step_size=float(eps_h[k]), numerical_error=int(nerr_h[k]),
                      n_steps=int(nst_h[k]), is_adapt=k < n_adapts) for k in range(n_samples)]  # step_size: mean over chains
        dl = []
        if keep_draws:
            dl = list(dr.unbind(0) if hasattr(dr, "unbind") else dr)
            if drop_warmup:
                dl = dl[n_adapts:]
        return SampleResult(zl.theta, dl, stats, eps, minv, int(nst_h.sum()), tm)
    draws, total_steps = [], 0
    acc, nerr, nst, eps_used, is_adapt = [], [], [], [], []  # per-iteration pooled scalars, fetched once at the end
    n_adapts = min(n_adapts, n_samples) if adaptor is not None else 0
    if n_adapts > 0:
        adaptor.initialize(n_adapts)
    minv_seen = None

    def one(i, adapting):
        nonlocal z, h, kappa, minv_seen
        t0 = time.perf_counter()
        tr = A.transition(rng, h, kappa, z)
        z = tr.z
        t1 = time.perf_counter()
        eps_used.append(A.step_size(kappa.tau.integrator))
        if adapting:  # Adaptation.adapt! glue (sampler.jl:72-90)
            kind = getattr(getattr(adaptor, "pc", None), "record_kind", "diag")
            rec = merge_records(allgather_records(iteration_record(z, tr.stat["acceptance_rate"], kind)), kind)
            adaptor.adapt(rec)
            if i == n_adapts:
                adaptor.finalize()
            if adaptor.Minv is not None and adaptor.Minv is not minv_seen:  # update(h, adaptor): only when it changed
                minv_seen = adaptor.Minv
                h = A.Hamiltonian(A.renew(h.metric, np.array(minv_seen)), h.target)
            tau = kappa.tau
            kappa = A.HMCKernel(A.Trajectory(tau.sampler, A.update_nom_step_size(tau.integrator, adaptor.eps),
                                             tau.termination_criterion), kappa.refreshment)
        t2 = time.perf_counter()
        acc.append(_mean(tr.stat["acceptance_rate"]))
        nerr.append(_sum(tr.stat["numerical_error"]))
        ns = tr.stat["n_steps"]
        nst.append(_sum(ns) if hasattr(ns, "sum") else int(ns) * theta.shape[0])
        is_adapt.append(adapting)
        if keep_draws and (not drop_warmup or not adapting):
            draws.append(z.theta.clone())
        t3 = time.perf_counter()
        tm["transition"] += t1 - t0
        tm["adapt"] += t2 - t1
        tm["bookkeeping"] += t3 - t2

    for i in range(1, n_adapts + 1):
        one(i, True)
    n_rest = n_samples - n_adapts
    fusable = (type(kappa.tau.integrator) is A.Leapfrog and
               (isinstance(kappa.tau.termination_criterion, A._DYNAMIC) or kappa.tau.sampler is A.EndPointTS))
    if n_rest > 0 and fused_sampling and isinstance(rng, A.PhiloxRNG) and fusable:
        t0 = time.perf_counter()
        z, dr, st = A.sample_transitions(rng, h, kappa, z, n_rest, keep_draws=keep_draws)
        if hasattr(z.theta, "is_cuda") and z.theta.is_cuda:
            torch.cuda.synchronize(z.theta.device)
        tm["sampling_launch"] += time.perf_counter() - t0
        a, e, n = st["acceptance_rate"], st["numerical_error"], st["n_steps"]
        if hasattr(a, "detach"):  # (T,) device vectors: one chunk each, fetched once below
            acc.append(a.double().mean(dim=1))
            nerr.append(e.sum(dim=1))
            nst.append(n.sum(dim=1))
        else:
            acc.extend(np.asarray(a, dtype=np.float64).mean(axis=1))
            nerr.extend(np.asarray(e).sum(axis=1))
            nst.extend(np.asarray(n).sum(axis=1))
        eps_used.extend([A.step_size(kappa.tau.integrator)] * n_rest)
        is_adapt.extend([False] * n_rest)
        if keep_draws:
            draws.extend(dr.unbind(0) if hasattr(dr, "unbind") else list(dr))
    else:
        for i in range(n_adapts + 1, n_samples + 1):
            one(i, False)

    t0 = time.perf_counter()

    def fetch(xs):  # one device->host transfer for the whole run (entries: 0-d scalars or (T,) chunks)
        if xs and hasattr(xs[0], "detach"):
            return torch.cat([x.double().reshape(-1) for x in xs]).cpu().numpy()
        return np.asarray([float(x) for x in xs], dtype=np.float64)

    acc_h, nerr_h, nst_h = fetch(acc), fetch(nerr), fetch(nst)
    stats = [dict(acceptance_rate=float(acc_h[k]), step_size=eps_used[k], numerical_error=int(nerr_h[k]),
                  n_steps=int(nst_h[k]), is_adapt=is_adapt[k]) for k in range(len(acc_h))]
    total_steps = int(nst_h.sum())
    tm["bookkeeping"] += time.perf_counter() - t0
    return SampleResult(z.theta, draws, stats, A.step_size(kappa.tau.integrator),
                        None if adaptor is None else adaptor.Minv, total_steps, tm)


# ------------------------------------------------------------------------------------------------ device-side pooling
class Comm:
    """`ahmc_comm`: the NCCL communicator of the ranks that share one adaptation.  `from_torch_distributed` creates it from
    the default process group (rank 0 draws the unique id, `broadcast_object_list` ships the 128 bytes)."""

    def __init__(self, ctx, handle, nranks, rank):
        self.ctx, self.h, self.nranks, self.rank = ctx, handle, nranks, rank

    @staticmethod
    def from_torch_distributed(device: int = 0) -> Optional["Comm"]:
        import ctypes as C

        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return None
        ctx = A.get_context(device)
        rank, world = dist.get_rank(), dist.get_world_size()
        buf = (C.c_char * 128)()
        if rank == 0:
            ctx.check(ctx.lib.ahmc_comm_unique_id(ctx.h, C.cast(buf, C.c_void_p)))
        box = [bytes(buf)]
        dist.broadcast_object_list(box, src=0)
        idb = C.create_string_buffer(box[0], 128)
        h = C.c_void_p()
        ctx.check(ctx.lib.ahmc_comm_create(ctx.h, C.cast(idb, C.c_void_p), world, rank, C.byref(h)))
        return Comm(ctx, h, world, rank)

    def allgather(self, record, flags: int = 0):
        """`ahmc_adapt_allgather_f64`: (n,) device tensor -> (nranks, n) device tensor, on the context stream."""
        import torch

        out = torch.empty((self.nranks, record.numel()), dtype=torch.float64, device=record.device)
        self.ctx.check(self.ctx.lib.ahmc_adapt_allgather_f64(self.ctx.h, self.h, record.data_ptr(), record.numel(),
                                                              out.data_ptr(), flags))
        return out

    def destroy(self):
        if self.h is not None:
            self.ctx.lib.ahmc_comm_destroy(self.ctx.h, self.h)
            self.h = None


class PooledDeviceAdaptor:
    """`ahmc_pooled`: StanHMCAdaptor(WelfordVar, NesterovDualAveraging) pooled over all chains of all ranks, resident on
    the device.  `eps` (N,) and `Minv` (D,) are torch views of the buffers the library updates in place -- hand them to
    `Leapfrog` / `DiagEuclideanMetric` once; `exchange` then needs no host work beyond one foreign call.
    `dense=True`: StanHMCAdaptor(WelfordCov, ...) (ahmc_pooled_create_dense, D <= 512); `Minv0` is (D, D), `Minv` and `cholU`
    (the upper factor U, U'U = Minv) are (D, D) views of the column-major device buffers -- hand them to
    `DenseEuclideanMetric(ad.Minv, cholU=ad.cholU)` once."""

    def __init__(self, device: int, D: int, N: int, n_adapts: int, eps0: float, delta: float = 0.8, adapt_metric: bool = True,
                 init_buffer: int = 75, term_buffer: int = 50, window_size: int = 25, gamma: float = 0.05, t0: float = 10.0,
                 kappa: float = 0.75, n_min: int = 10, Minv0=None, dense: bool = False):
        import ctypes as C

        import torch

        from . import _lib as L

        self.ctx = ctx = A.get_context(device)
        self.D, self.N, self.n_adapts, self.dense = D, N, n_adapts, dense
        cfg = L.PooledCfg(n_adapts, init_buffer, term_buffer, window_size, delta, gamma, t0, kappa, float(eps0),
                          1 if adapt_metric else 0, n_min)
        m0 = None if Minv0 is None else np.ascontiguousarray(Minv0, dtype=np.float64)
        if dense and m0 is not None:
            if m0.shape != (D, D):
                raise L.InvalidArgument(L.ERR_INVALID, f"Minv0 must be ({D}, {D}), got {m0.shape}")
            m0 = np.ascontiguousarray(m0.T)  # column-major
        self.h = C.c_void_p()
        create = ctx.lib.ahmc_pooled_create_dense if dense else ctx.lib.ahmc_pooled_create
        ctx.check(create(ctx.h, D, N, C.byref(cfg), None if m0 is None else m0.ctypes.data_as(L._dp), C.byref(self.h)))
        dev = torch.device("cuda", device)
        self.eps = torch.as_tensor(A._RawCuda(ctx.lib.ahmc_pooled_eps(self.h), (N,)), device=dev)
        if dense:  # a row-major (D, D) view of a column-major buffer is the transpose: present the logical matrices
            self.Minv = torch.as_tensor(A._RawCuda(ctx.lib.ahmc_pooled_minv(self.h), (D, D)), device=dev).T
            self.cholU = torch.as_tensor(A._RawCuda(ctx.lib.ahmc_pooled_cholu(self.h), (D, D)), device=dev).T
        else:
            self.Minv = torch.as_tensor(A._RawCuda(ctx.lib.ahmc_pooled_minv(self.h), (D,)), device=dev)

    def exchange(self, theta, acceptance_rate, comm: Optional[Comm] = None, eps_trace=None, flags: int = A.L.FLAG_ASYNC):
        """`adapt!` of the next iteration (ahmc_adapt_exchange_f64): K5 -> all-gather -> merge + adaptor update, on the stream"""
        self.ctx.check(self.ctx.lib.ahmc_adapt_exchange_f64(self.ctx.h, None if comm is None else comm.h, self.h, self.D, self.N,
                                                             theta.data_ptr(), self.D, acceptance_rate.data_ptr(),
                                                             None if eps_trace is None else eps_trace.data_ptr(), flags))

    def state(self):
        """synchronising read-back -> dict(eps, Minv, iteration, merged_record); a dense adaptor adds cholU (U) and
        failed_iteration (the first iteration whose estimate was not positive definite, 0 = none)"""
        import ctypes as C

        from . import _lib as L

        eps, it = C.c_double(), C.c_int32()
        if self.dense:
            D = self.D
            failed = C.c_int32()
            minv, U, rec = np.empty((D, D)), np.empty((D, D)), np.empty(2 + 2 * D + D * D)
            self.ctx.check(self.ctx.lib.ahmc_pooled_state_dense(self.ctx.h, self.h, C.byref(eps), minv.ctypes.data_as(L._dp),
                                                                 U.ctypes.data_as(L._dp), C.byref(it), rec.ctypes.data_as(L._dp),
                                                                 C.byref(failed)))
            return dict(eps=eps.value, Minv=np.ascontiguousarray(minv.T), cholU=np.ascontiguousarray(U.T), iteration=it.value,
                        merged_record=rec, failed_iteration=failed.value)
        minv, rec = np.empty(self.D), np.empty(2 + 2 * self.D)
        self.ctx.check(self.ctx.lib.ahmc_pooled_state(self.ctx.h, self.h, C.byref(eps), minv.ctypes.data_as(L._dp), C.byref(it),
                                                       rec.ctypes.data_as(L._dp)))
        return dict(eps=eps.value, Minv=minv, iteration=it.value, merged_record=rec)

    def destroy(self):
        if self.h is not None:
            self.ctx.lib.ahmc_pooled_destroy(self.ctx.h, self.h)
            self.h = None


def sample_pooled_device(rng, h: A.Hamiltonian, kappa: A.HMCKernel, theta, n_samples: int, n_adapts: int, eps0: float,
                         delta: float = 0.8, adapt_metric: bool = True, comm: Optional[Comm] = None, windows=(75, 50, 25),
                         keep_eps_trace: bool = False) -> SampleResult:
    """`sample` with the pooled StanHMCAdaptor on the DEVICE: every warm-up iteration is [transition kernel, K5, all-gather,
    adaptor-update kernel] enqueued on one stream -- no device->host copy, no synchronisation, no new Hamiltonian / kernel
    objects; the sampling phase is the persistent launch.  Dynamic (NUTS) and fixed-n static trajectories (a
    FixedIntegrationTime trajectory needs eps on the host to size the trajectory: use `sample`).
    A DenseEuclideanMetric adapts with the pooled WelfordCov (D <= 512): M^-1 and its Cholesky factor are replaced on the
    device at window ends; an estimate that is not positive definite raises AhmcError after the warm-up, naming the iteration."""
    import time

    import torch

    dense = isinstance(h.metric, A.DenseEuclideanMetric)
    if not (dense or isinstance(h.metric, A.DiagEuclideanMetric)):
        raise A.L.AhmcError(A.L.ERR_UNSUPPORTED,
                            "pooled device adaptation: DiagEuclideanMetric (WelfordVar) or DenseEuclideanMetric (WelfordCov)")
    tau = kappa.tau
    if isinstance(tau.termination_criterion, A.FixedIntegrationTime):
        raise A.L.AhmcError(A.L.ERR_UNSUPPORTED, "FixedIntegrationTime needs eps on the host; use sample()")
    N, D = theta.shape
    dev = theta.device
    tm = dict(transition=0.0, adapt=0.0, sampling_launch=0.0, bookkeeping=0.0)
    n_adapts = min(n_adapts, n_samples)
    Minv0 = h.metric.Minv if A._is_host(h.metric.Minv) else h.metric.Minv.detach().cpu().numpy()
    ad = PooledDeviceAdaptor(dev.index or 0, D, N, n_adapts, eps0, delta, adapt_metric, *windows, Minv0=Minv0, dense=dense)
    hd = A.Hamiltonian(A.DenseEuclideanMetric(ad.Minv, cholU=ad.cholU) if dense else A.DiagEuclideanMetric(ad.Minv), h.target)
    if isinstance(tau.integrator, A.JitteredLeapfrog):
        raise A.L.AhmcError(A.L.ERR_UNSUPPORTED, "JitteredLeapfrog draws its step size on the host; use sample()")
    lf_d = A.TemperedLeapfrog(ad.eps, tau.integrator.alpha) if isinstance(tau.integrator, A.TemperedLeapfrog) else A.Leapfrog(ad.eps)
    kd = A.HMCKernel(A.Trajectory(tau.sampler, lf_d, tau.termination_criterion), kappa.refreshment)
    z = A.phasepoint(hd, theta, torch.zeros_like(theta))
    acc, nerr, nst = [], [], []
    t0 = time.perf_counter()
    # torch work (allocation / release of the per-iteration buffers, the scalar reductions) runs on the CONTEXT's stream:
    # the transition and exchange calls are asynchronous, so everything that touches their buffers must be ordered with them
    torch.cuda.current_stream(dev).synchronize()
    with torch.cuda.stream(ad.ctx.torch_stream()):
        trace = torch.zeros(max(n_adapts, 1), dtype=torch.float64, device=dev) if keep_eps_trace else None
        for _ in range(n_adapts):
            tr = A.transition(rng, hd, kd, z, flags=A.L.FLAG_ASYNC)
            z = tr.z
            ad.exchange(z.theta, tr.stat["acceptance_rate"], comm, trace)
            acc.append(tr.stat["acceptance_rate"].mean())
            nerr.append(tr.stat["numerical_error"].sum())
            nst.append(tr.stat["n_steps"].sum())
        tm["issue_warmup"] = time.perf_counter() - t0
        torch.cuda.synchronize(dev)
    tm["transition"] = time.perf_counter() - t0  # warm-up wall time: transitions and exchanges share one stream
    if dense and n_adapts > 0:
        failed = ad.state()["failed_iteration"]
        if failed:
            ad.destroy()
            raise A.L.AhmcError(A.L.ERR_INVALID, f"pooled WelfordCov: the adapted M^-1 of warm-up iteration {failed} is not "
                                                 "positive definite (Cholesky failed); M^-1 and its factor kept their previous value")
    n_rest = n_samples - n_adapts
    draws = []
    if n_rest > 0:
        t1 = time.perf_counter()
        z, dr, st = A.sample_transitions(rng, hd, kd, z, n_rest, keep_draws=False)
        torch.cuda.synchronize(dev)
        tm["sampling_launch"] = time.perf_counter() - t1
        acc.append(st["acceptance_rate"].double().mean(dim=1))
        nerr.append(st["numerical_error"].sum(dim=1))
        nst.append(st["n_steps"].sum(dim=1))
    cat = lambda xs: torch.cat([x.double().reshape(-1) for x in xs]).cpu().numpy() if xs else np.zeros(0)
    acc_h, nerr_h, nst_h = cat(acc), cat(nerr), cat(nst)
    s = ad.state()
    stats = [dict(acceptance_rate=float(acc_h[k]), step_size=None, numerical_error=int(nerr_h[k]), n_steps=int(nst_h[k]),
                  is_adapt=k < n_adapts) for k in range(len(acc_h))]
    if keep_eps_trace:
        tr_h = trace.cpu().numpy()
        for k in range(n_adapts):
            stats[k]["step_size_after"] = float(tr_h[k])
    res = SampleResult(z.theta, draws, stats, s["eps"], s["Minv"], int(nst_h.sum()), tm)
    ad.destroy()
    return res
