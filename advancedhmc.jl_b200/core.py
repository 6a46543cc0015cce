"""core.py -- host-side mirror of AdvancedHMC.jl's plugin surface for the leapfrog / HMC / NUTS path,
above the C ABI of libahmc_b200 (include/ahmc_b200.h).

Julia is not available in this image, so the host side the north star asks for ("Julia host code keeps
the AbstractIntegrator / Hamiltonian / AbstractMetric plugin surface and calls through a thin ccall
layer") is mirrored here in Python with the same names, argument meaning and error behaviour; the Julia
shim itself is julia/AdvancedHMCB200Ext.jl (unexecuted).  Citations: /root/reference/<file>:<line>.

Array convention: Julia's column-major `D x N` matrix is byte-identical to a C-contiguous `(N, D)`
array, so every position / momentum / gradient here is a float64 array of shape (N, D) -- a CUDA
`torch.Tensor` (device-pointer calls) or a `numpy.ndarray` (AHMC_FLAG_HOST_BUFFERS calls: the library
stages host<->device itself).  A 1-D array of length D is a single chain (the reference's vector mode).
PyTorch is used for device memory and streams only; all arithmetic happens in the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field, replace
from typing import Any, Optional, Sequence, Union

import numpy as np

from . import _lib as L

try:  # torch is plumbing (device memory); host-buffer mode works without a tensor in sight
    import torch
except Exception:  # pragma: no cover
    torch = None

Array = Any

# ------------------------------------------------------------------------------------------------
# context
# ------------------------------------------------------------------------------------------------
_contexts: dict = {}


class Context:
    """One `ahmc_ctx` per device (created lazily; bound to its own non-blocking stream)."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        self.lib = L.load()
        self.device = device
        self.stream = stream  # raw cudaStream_t the context is bound to (None: its own stream)
        h = C.c_void_p()
        rc = self.lib.ahmc_create(C.byref(h), device, C.c_void_p(stream) if stream else None)
        if rc != L.OK:
            raise RuntimeError(
                f"ahmc_create(device={device}) failed with code {rc}: libahmc_b200 needs a CUDA device "
                "(there is no CPU fallback; the CPU restatement under oracle/ is test infrastructure only)")
        self.h = h

    def check(self, rc: int):
        if rc == L.OK:
            return
        msg = self.lib.ahmc_last_error(self.h).decode()
        if rc == L.ERR_INVALID:
            raise L.InvalidArgument(rc, msg)
        raise L.AhmcError(rc, msg)

    @property
    def launches(self) -> int:
        return int(self.lib.ahmc_launch_count(self.h))

    def synchronize(self):
        self.check(self.lib.ahmc_synchronize(self.h))

    def torch_stream(self):
        """the context's stream as a torch stream: run torch work that feeds / consumes FLAG_ASYNC calls under
        `with torch.cuda.stream(ctx.torch_stream())` so that torch's allocator and kernels are ordered with ours"""
        return torch.cuda.ExternalStream(int(self.lib.ahmc_stream(self.h)), device=torch.device("cuda", self.device))

    def last_transport(self) -> str:
        """how the last host-buffer `step` moved its buffers (ahmc_last_transport)"""
        return self.lib.ahmc_last_transport(self.h).decode()


def get_context(device: int = 0, stream: Optional[int] = None) -> Context:
    """The process-wide context of `device`.  Pass `stream` (a raw cudaStream_t, e.g.
    torch.cuda.Stream().cuda_stream) on the FIRST call to bind the context to that stream."""
    if device not in _contexts:
        _contexts[device] = Context(device, stream)
    return _contexts[device]


def _is_host(x) -> bool:
    return isinstance(x, np.ndarray)


def _ptr(x) -> Optional[int]:
    if x is None:
        return None
    if _is_host(x):
        return x.ctypes.data
    return x.data_ptr()


def _check_arr(x, name, dtype=np.float64):
    if _is_host(x):
        if x.dtype != dtype or not x.flags["C_CONTIGUOUS"]:
            raise L.InvalidArgument(L.ERR_INVALID, f"{name} must be a C-contiguous {np.dtype(dtype).name} array")
    else:
        if torch is None or not isinstance(x, torch.Tensor):
            raise L.InvalidArgument(L.ERR_INVALID, f"{name} must be a numpy array or a CUDA torch tensor")
        if not x.is_cuda or not x.is_contiguous():
            raise L.InvalidArgument(L.ERR_INVALID, f"{name} must be a contiguous CUDA tensor")
    return x


def _like(x, shape, dtype=np.float64):
    if _is_host(x):
        return np.empty(shape, dtype=dtype)
    tdt = {np.float64: torch.float64, np.int32: torch.int32, np.uint8: torch.uint8, np.uint32: torch.int32}[dtype]
    return torch.empty(shape, dtype=tdt, device=x.device)


def _device_of(x) -> int:
    if _is_host(x):
        return torch.cuda.current_device() if (torch is not None and torch.cuda.is_available()) else 0
    return x.device.index or 0


def _sync_torch(x):
    """Inputs produced on torch's current stream must be complete before our context stream reads them
    (no-op when the context is bound to that very stream)."""
    if not _is_host(x) and torch is not None:
        cur = torch.cuda.current_stream(x.device)
        ctx = _contexts.get(x.device.index or 0)
        if ctx is None or ctx.stream != cur.cuda_stream:
            cur.synchronize()


# ------------------------------------------------------------------------------------------------
# targets: the (lp, dlp/dtheta) closures of `Hamiltonian` (src/hamiltonian.jl:1-6), built in
# ------------------------------------------------------------------------------------------------
class _Target:
    kind: int
    D: int

    def __init__(self, kind, D, p0=None, p1=None, c0=0.0):
        self.kind, self.D, self.c0 = kind, int(D), float(c0)
        self.p0 = None if p0 is None else np.ascontiguousarray(p0, dtype=np.float64)
        self.p1 = None if p1 is None else np.ascontiguousarray(p1, dtype=np.float64)
        self._handles: dict = {}

    def handle(self, ctx: Context):
        h = self._handles.get(ctx.device)
        if h is None:
            h = C.c_void_p()
            p0 = None if self.p0 is None else self.p0.ctypes.data_as(C.POINTER(C.c_double))
            p1 = None if self.p1 is None else self.p1.ctypes.data_as(C.POINTER(C.c_double))
            ctx.check(ctx.lib.ahmc_model_create(ctx.h, self.kind, self.D, p0, p1, self.c0, C.byref(h)))
            self._handles[ctx.device] = h
        return h


class StdNormal(_Target):
    """lp(theta) = c0 - sum(theta^2)/2   (the `NegU` / unit Gaussian targets of test/integrator.jl:109-117)."""

    def __init__(self, D, c0=0.0):
        super().__init__(L.MODEL_STD_NORMAL, D, c0=c0)


class DiagGaussian(_Target):
    """Independent N(m, s^2): the hand-coded Gaussian of test/common.jl:35-77 (with the true gradient).
    `normalised=True` adds the -sum(log(2 pi) + 2 log s)/2 constant that test/common.jl:40-42 includes."""

    def __init__(self, m, s, normalised=True):
        m, s = np.asarray(m, dtype=np.float64), np.asarray(s, dtype=np.float64)
        if m.shape != s.shape or m.ndim != 1:
            raise L.InvalidArgument(L.ERR_INVALID, "m and s must be vectors of equal length")
        c0 = float(-0.5 * np.sum(np.log(2 * np.pi) + 2 * np.log(s))) if normalised else 0.0
        super().__init__(L.MODEL_DIAG_GAUSS, m.size, m, s, c0)


class DenseGaussian(_Target):
    """Correlated Gaussian with precision matrix P: lp = c0 - (theta-mu)' P (theta-mu) / 2."""

    def __init__(self, mu, P, c0=0.0):
        mu, P = np.asarray(mu, dtype=np.float64), np.asarray(P, dtype=np.float64)
        if P.shape != (mu.size, mu.size):
            raise L.InvalidArgument(L.ERR_INVALID, "P must be D x D")
        super().__init__(L.MODEL_DENSE_GAUSS, mu.size, mu, np.ascontiguousarray(P.T), c0)


class Funnel(_Target):
    """Neal's funnel: theta_1 ~ N(0, 3), theta_i ~ N(0, exp(theta_1 / 2)) (std), i > 1."""

    def __init__(self, D, c0=0.0):
        super().__init__(L.MODEL_FUNNEL, D, c0=c0)


class UserTarget(_Target):
    """A user-supplied log pi / grad log pi as CUDA source, compiled at run time INTO the fused kernels
    (ahmc_model_create_user; the `h.dlp/dtheta` closure of src/hamiltonian.jl:45-48 as a device function).  `source` defines
    `__device__ double ahmc_user_logp_grad(const double* theta, double* grad, int D, const double* params)` (PLUS gradient)
    or, with `#define AHMC_USER_COORDWISE`, `__device__ double ahmc_user_coord(int d, double theta_d, const double* params,
    double* grad_d)`.  Works with phasepoint, step, static HMC transitions, NUTS and find_good_stepsize_batched."""

    def __init__(self, D: int, source: str, params=None, c0: float = 0.0):
        self.kind, self.D, self.c0 = L.MODEL_USER, int(D), float(c0)
        self.source = source
        self.params = None if params is None else np.ascontiguousarray(params, dtype=np.float64).reshape(-1)
        self._handles = {}

    def handle(self, ctx: "Context"):
        h = self._handles.get(ctx.device)
        if h is None:
            h = C.c_void_p()
            p = self.params
            ctx.check(ctx.lib.ahmc_model_create_user(ctx.h, self.D, self.source.encode(), None if p is None else p.ctypes.data_as(L._dp),
                                                     0 if p is None else p.size, self.c0, C.byref(h)))
            self._handles[ctx.device] = h
        return h

    @staticmethod
    def check_source(source: str, D: int, kernel: int = 1, metric_kind: int = 1):
        """compile-only check (no GPU needed): raises InvalidArgument with the NVRTC log if `source` does not compile"""
        log = C.create_string_buffer(8192)
        rc = L.load().ahmc_user_source_check(source.encode(), kernel, metric_kind, D, log, 8192)
        if rc != L.OK:
            raise L.InvalidArgument(rc, log.value.decode())


class _RawCuda:
    """zero-copy view of a raw device pointer for torch (via __cuda_array_interface__)."""

    def __init__(self, ptr, shape):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": "<f8", "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class CallbackTarget(_Target):
    """An arbitrary user log-density: `fn(theta) -> (lp, grad)` on CUDA tensors, theta of shape (N, D), lp (N,),
    grad (N, D) = PLUS gradient of log pi -- the role of the `lp` / `dlp/dtheta` closures of `Hamiltonian`
    (src/hamiltonian.jl:1-6, 45-48).  The engine runs in split-step mode: per leapfrog step two small fused kernels
    with `fn` evaluated in between on the context's stream (any torch code, autograd included).  Supported by
    phasepoint / step / static-HMC transition; NUTS needs a device-resident (built-in) target."""

    def __init__(self, D, fn):
        self.kind, self.D, self.c0, self.p0, self.p1 = L.MODEL_CALLBACK, int(D), 0.0, None, None
        self.fn = fn
        self._handles = {}
        self.error = None
        self._cfn = L.LOGP_GRAD_FN(self._trampoline)

    def _trampoline(self, user, theta, lp, grad, D, N, ld, stream):
        try:
            dev = torch.device("cuda", torch.cuda.current_device())
            view = lambda p, shape: torch.as_tensor(_RawCuda(p, shape), device=dev)
            with torch.cuda.stream(torch.cuda.ExternalStream(int(stream))):
                th = view(theta, (N, ld))[:, :D]
                v, g = self.fn(th)
                view(lp, (N,)).copy_(v)
                view(grad, (N, ld))[:, :D].copy_(g)
            return 0
        except Exception as e:  # never raise across the C ABI
            self.error = e
            return 1

    def handle(self, ctx: Context):
        h = self._handles.get(ctx.device)
        if h is None:
            h = C.c_void_p()
            ctx.check(ctx.lib.ahmc_model_create_callback(ctx.h, self.D, self._cfn, None, C.byref(h)))
            self._handles[ctx.device] = h
        return h


# ------------------------------------------------------------------------------------------------
# metrics (src/metric.jl)
# ------------------------------------------------------------------------------------------------
class AbstractMetric:
    pass


class GaussianKinetic:
    pass


class UnitEuclideanMetric(AbstractMetric):
    """src/metric.jl:17-35.  `size` = (D,) or (D, N)."""

    kind = L.METRIC_UNIT

    def __init__(self, size):
        self.size = (size,) if isinstance(size, int) else tuple(size)
        self.Minv = None

    def _desc(self, D, N, like):
        return L.Metric(L.METRIC_UNIT, None, 0, None), ()


class DiagEuclideanMetric(AbstractMetric):
    """src/metric.jl:52-72.  Minv: (D,) shared, or (N, D) per chain (Julia's D x N form, :64)."""

    kind = L.METRIC_DIAG

    def __init__(self, Minv):
        if isinstance(Minv, (int, tuple)):
            sz = (Minv,) if isinstance(Minv, int) else tuple(Minv)
            Minv = np.ones(sz[0]) if len(sz) == 1 else np.ones((sz[1], sz[0]))
        self.Minv = Minv
        self.size = tuple(Minv.shape) if Minv.ndim == 1 else (Minv.shape[1], Minv.shape[0])

    @property
    def sqrtMinv(self):
        return np.sqrt(self.Minv) if _is_host(self.Minv) else self.Minv.sqrt()

    def _desc(self, D, N, like):
        Mi = _coerce_like(self.Minv, like)
        if Mi.shape[-1] != D or (Mi.ndim == 2 and Mi.shape[0] != N):
            raise L.InvalidArgument(L.ERR_INVALID, f"AxesMismatch: Minv has shape {tuple(Mi.shape)} but r is ({N},{D})")
        stride = D if Mi.ndim == 2 else 0
        return L.Metric(L.METRIC_DIAG, _ptr(Mi), stride, None), (Mi,)


class DenseEuclideanMetric(AbstractMetric):
    """src/metric.jl:89-120.  Minv: (D, D); cholU = cholesky(Symmetric(Minv)).U (host LAPACK via numpy).
    `cholU=` hands over the upper factor instead (U'U = Minv, both (D, D) as logical matrices): with CUDA tensors nothing is
    copied to the host or factorised there and device calls read the two tensors in place (e.g. the buffers of a dense
    `PooledDeviceAdaptor`, which change under the metric at window ends)."""

    kind = L.METRIC_DENSE

    def __init__(self, Minv, cholU=None):
        if isinstance(Minv, int):
            Minv = np.eye(Minv)
        self.Minv, self.cholU = Minv, cholU
        if cholU is not None:
            if tuple(Minv.shape) != tuple(cholU.shape) or Minv.ndim != 2:
                raise L.InvalidArgument(L.ERR_INVALID, "Minv and cholU must both be D x D")
            self.size = (Minv.shape[0],)
            return
        Mh = Minv if _is_host(Minv) else Minv.detach().cpu().numpy()
        self._Minv_h = np.ascontiguousarray(Mh, dtype=np.float64)
        self._cholU_h = np.ascontiguousarray(np.linalg.cholesky(self._Minv_h).T)  # upper factor
        self.size = (Mh.shape[0],)

    def _desc(self, D, N, like):
        if self.cholU is not None:
            if self.size != (D,):
                raise L.InvalidArgument(L.ERR_INVALID, f"AxesMismatch: Minv is {self.size * 2} but r has {D} rows")
            # column-major D x D == row-major transpose; a tensor whose transpose is contiguous (the adaptor's views) is
            # passed as it is
            Mi, U = (_colmajor(x, like) for x in (self.Minv, self.cholU))
            return L.Metric(L.METRIC_DENSE, _ptr(Mi), 0, _ptr(U)), (Mi, U)
        if self._Minv_h.shape != (D, D):
            raise L.InvalidArgument(L.ERR_INVALID, f"AxesMismatch: Minv is {self._Minv_h.shape} but r has {D} rows")
        # column-major D x D == transposed row-major; Minv symmetric, U stored column-major
        Mi = _coerce_like(np.ascontiguousarray(self._Minv_h.T), like)
        U = _coerce_like(np.ascontiguousarray(self._cholU_h.T), like)
        return L.Metric(L.METRIC_DENSE, _ptr(Mi), 0, _ptr(U)), (Mi, U)


def _colmajor(a, like):
    """the column-major buffer of the D x D matrix `a` at the residency of `like`"""
    if not _is_host(like) and not _is_host(a) and a.device == like.device and a.dtype == torch.float64 and a.T.is_contiguous():
        return a.T
    return _coerce_like(a.T if _is_host(a) else a.T.contiguous(), like)


def _coerce_like(a, like):
    """bring a parameter array to the residency of `like` (numpy -> host call, torch -> device call)."""
    if _is_host(like):
        return np.ascontiguousarray(a if _is_host(a) else a.detach().cpu().numpy(), dtype=np.float64)
    if _is_host(a):
        return torch.as_tensor(a, dtype=torch.float64, device=like.device).contiguous()
    return a.to(like.device, torch.float64).contiguous()


def renew(metric: AbstractMetric, Minv) -> AbstractMetric:
    """src/metric.jl:31,69,117."""
    if isinstance(metric, UnitEuclideanMetric):
        return UnitEuclideanMetric(metric.size)
    return type(metric)(Minv)


# ------------------------------------------------------------------------------------------------
# Hamiltonian / PhasePoint (src/hamiltonian.jl)
# ------------------------------------------------------------------------------------------------
@dataclass
class Hamiltonian:
    """src/hamiltonian.jl:1-6.  `target` plays the role of the (lp, dlp/dtheta) closure pair."""

    metric: AbstractMetric
    target: _Target
    kinetic: GaussianKinetic = field(default_factory=GaussianKinetic)


@dataclass
class DualValue:
    """src/hamiltonian.jl:22-38."""

    value: Array
    gradient: Array


class PhasePoint:
    """src/hamiltonian.jl:88-107.  lp.gradient holds MINUS grad log pi (hamiltonian.jl:45-48)."""

    __slots__ = ("theta", "r", "lp", "lk")

    def __init__(self, theta, r, lp: DualValue, lk: DualValue):
        n = tuple(theta.shape)
        # lp.gradient may be None: "not cached" -- `step` then recomputes it on the device for built-in targets
        if (tuple(r.shape) != n or (lp.gradient is not None and tuple(lp.gradient.shape) != n)
                or (lk.gradient is not None and tuple(lk.gradient.shape) != n)):
            raise L.InvalidArgument(L.ERR_INVALID, "length(theta) == length(r) == length(lp.gradient) == length(lk.gradient) violated")
        self.theta, self.r, self.lp, self.lk = theta, r, lp, lk

    def _nd(self):
        return (1, self.theta.shape[0]) if self.theta.ndim == 1 else tuple(self.theta.shape)

    def _c(self, with_lk_gradient=True):
        N, D = self._nd()
        return L.PhasePoint(_ptr(self.theta), _ptr(self.r), _ptr(self.lp.value), _ptr(self.lp.gradient),
                            _ptr(self.lk.value), _ptr(self.lk.gradient) if with_lk_gradient else None, D)

    def isfinite(self):
        """Base.isfinite(z) (hamiltonian.jl:141-142) -- over ALL chains, like the reference."""
        xs = [self.lp.value, self.lp.gradient, self.lk.value] + ([self.lk.gradient] if self.lk.gradient is not None else [])
        if _is_host(self.theta):
            return bool(all(np.all(np.isfinite(x)) for x in xs))
        return bool(all(torch.isfinite(x).all().item() for x in xs))


def _empty_pp(like, with_lk_gradient=True):
    shp = tuple(like.shape)
    nshp = shp[:-1] if like.ndim == 2 else ()
    v = lambda: _like(like, nshp if nshp else (1,))
    return PhasePoint(_like(like, shp), _like(like, shp), DualValue(v(), _like(like, shp)),
                      DualValue(v(), _like(like, shp) if with_lk_gradient else None))


def neg_energy(z: PhasePoint):
    """hamiltonian.jl:149."""
    return z.lp.value + z.lk.value


def energy(z: PhasePoint):
    """hamiltonian.jl:194."""
    return -neg_energy(z)


def phasepoint(h: Hamiltonian, theta, r, flags: int = 0) -> PhasePoint:
    """phasepoint(h, theta, r) (hamiltonian.jl:115-119) -> ahmc_phasepoint_f64."""
    _check_arr(theta, "theta"), _check_arr(r, "r")
    if tuple(theta.shape) != tuple(r.shape):
        raise L.InvalidArgument(L.ERR_INVALID, "theta and r must have the same shape")
    ctx = get_context(_device_of(theta))
    z = _empty_pp(theta)
    z.theta, z.r = theta, r
    N, D = z._nd()
    md, keep = h.metric._desc(D, N, theta)
    _sync_torch(theta)
    zc = z._c()
    ctx.check(ctx.lib.ahmc_phasepoint_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, C.byref(zc),
                                          flags | (L.FLAG_HOST_BUFFERS if _is_host(theta) else 0)))
    return z


def dHdr(h: Hamiltonian, r):
    """dH/dr (hamiltonian.jl:50-68): lk.gradient of a phase point at r."""
    z = phasepoint(h, _like(r, tuple(r.shape)) * 0 if not _is_host(r) else np.zeros_like(r), r)
    return z.lk.gradient


# ------------------------------------------------------------------------------------------------
# RNG inputs
# ------------------------------------------------------------------------------------------------
class PhiloxRNG:
    """Counter-based generator living on the device (Philox4x32-10 keyed by seed; one `offset` tick per
    transition).  Replaces the reference's `AbstractRNG` / vector of RNGs (src/utilities.jl:5-23)."""

    def __init__(self, seed: int = 0):
        self.seed, self.offset = int(seed) & (2**64 - 1), 0

    def _c(self, advance=True):
        r = L.Rng(self.seed, self.offset, None, None, 0, None, 0, 0.0)
        if advance:
            self.offset += 1
        return r, ()

    def draw_n_fwd(self, n_steps: int) -> int:
        """the coupled `rand(0:n_steps)` of the multinomial-static transition (host side, one value for all chains)."""
        return int(np.random.Generator(np.random.Philox(key=self.seed, counter=[0, 0, 0, self.offset])).integers(0, n_steps + 1))


class TapeRNG:
    """Explicit random tapes: makes a transition a pure function (how parity with the oracle is defined).
    normal: (N, D); exp: (N,) static HMC or (N, n_exp) NUTS; dirs: (N, n_dir) uint8."""

    def __init__(self, normal=None, exp=None, dirs=None, n_fwd=None):
        self.normal, self.exp, self.dirs, self.n_fwd = normal, exp, dirs, n_fwd

    def draw_n_fwd(self, n_steps: int) -> int:
        if self.n_fwd is None:
            raise L.InvalidArgument(L.ERR_INVALID, "TapeRNG needs n_fwd for a MultinomialTS static transition")
        return int(self.n_fwd)

    def _c(self, advance=True):
        es = 1 if (self.exp is None or self.exp.ndim == 1) else self.exp.shape[1]
        ds = 0 if self.dirs is None else self.dirs.shape[1]
        return L.Rng(0, 0, _ptr(self.normal), _ptr(self.exp), es, _ptr(self.dirs), ds, 0.0), (self.normal, self.exp, self.dirs)


def rand_momentum(rng, metric: AbstractMetric, kinetic, theta):
    """rand_momentum(rng, metric, kinetic, theta) (metric.jl:290-320)."""
    ctx = get_context(_device_of(theta))
    r = _like(theta, tuple(theta.shape))
    N, D = (1, theta.shape[0]) if theta.ndim == 1 else tuple(theta.shape)
    md, keep = metric._desc(D, N, theta)
    rc, keep2 = rng._c()
    _sync_torch(theta)
    ctx.check(ctx.lib.ahmc_rand_momentum_f64(ctx.h, C.byref(md), D, N, C.byref(rc), _ptr(r), D,
                                             L.FLAG_HOST_BUFFERS if _is_host(theta) else 0))
    return r


# ------------------------------------------------------------------------------------------------
# integrators (src/integrator.jl)
# ------------------------------------------------------------------------------------------------
class AbstractIntegrator:
    pass


class AbstractLeapfrog(AbstractIntegrator):
    pass


@dataclass(frozen=True)
class Leapfrog(AbstractLeapfrog):
    """src/integrator.jl:71-74.  eps: float, or a per-chain array of length N (`AbstractScalarOrVec`)."""

    eps: Any


@dataclass(frozen=True)
class JitteredLeapfrog(AbstractLeapfrog):
    """src/integrator.jl:112-121."""

    eps0: Any
    jitter: float
    eps: Any = None

    def __post_init__(self):
        if self.eps is None:
            object.__setattr__(self, "eps", self.eps0)


@dataclass(frozen=True)
class TemperedLeapfrog(AbstractLeapfrog):
    """src/integrator.jl:174-179."""

    eps: Any
    alpha: float


def step_size(lf):  # integrator.jl:51
    return lf.eps


def nom_step_size(lf):  # integrator.jl:32, :136
    return lf.eps0 if isinstance(lf, JitteredLeapfrog) else lf.eps


def update_nom_step_size(lf, eps):  # integrator.jl:60, :138
    return replace(lf, eps0=eps) if isinstance(lf, JitteredLeapfrog) else replace(lf, eps=eps)


def stat(lf):  # integrator.jl:58
    return dict(step_size=step_size(lf), nom_step_size=nom_step_size(lf))


def jitter(rng: np.random.Generator, lf):
    """integrator.jl:52, :140-156: eps = eps0 * (1 + jitter * (2u - 1)), u ~ U(0,1) per chain."""
    if not isinstance(lf, JitteredLeapfrog):
        return lf
    e0 = lf.eps0
    if np.ndim(e0) == 0:
        return replace(lf, eps=e0 * (1 + lf.jitter * (2 * rng.random() - 1)))
    e0h = e0 if _is_host(e0) else e0.detach().cpu().numpy()
    e = e0h * (1 + lf.jitter * (2 * rng.random(e0h.shape) - 1))
    return replace(lf, eps=e if _is_host(e0) else torch.as_tensor(e, device=e0.device))


def temper(lf, r, step: tuple, n_steps: int):
    """integrator.jl:198-209; step = (i, is_half)."""
    if not isinstance(lf, TemperedLeapfrog):
        return r
    i, is_half = step
    if i > n_steps:
        raise IndexError("Current leapfrog iteration exceeds the total number of steps.")  # BoundsError
    i_temper = 2 * (i - 1) + 1 + (0 if is_half else 1)
    return r * math.sqrt(lf.alpha) if i_temper <= n_steps else r / math.sqrt(lf.alpha)


def _eps_args(eps, like, N):
    if np.ndim(eps) == 0:
        return float(eps), None, None
    e = _coerce_like(eps, like)
    if tuple(e.shape) != (N,):
        raise L.InvalidArgument(L.ERR_INVALID, f"per-chain step size must have length N={N}")
    return 0.0, _ptr(e), e


@dataclass
class StepInfo:
    status: Array
    steps_done: Array


def step(lf: AbstractLeapfrog, h: Hamiltonian, z: PhasePoint, n_steps: int = 1, *, fwd: Optional[bool] = None,
         flags: int = 0, return_info: bool = False, with_lk_gradient: bool = True,
         out: Optional[PhasePoint] = None, full_trajectory: bool = False):
    """`step(lf, h, z, n_steps; fwd)` (integrator.jl:216-265) -> ahmc_leapfrog_f64.
    Functional like the reference: returns a fresh PhasePoint, z is untouched."""
    if fwd is not None:
        n_steps = abs(n_steps) if fwd else -abs(n_steps)
    for nm in ("theta", "r"):
        _check_arr(getattr(z, nm), nm)
    if full_trajectory:
        return _step_full_trajectory(lf, h, z, n_steps, flags)
    ctx = get_context(_device_of(z.theta))
    N, D = z._nd()
    if out is None:
        out = _empty_pp(z.theta, with_lk_gradient)  # functional like the reference: fresh arrays
    else:
        with_lk_gradient = out.lk.gradient is not None
    status = _like(z.theta, (N,), np.uint32)
    done = _like(z.theta, (N,), np.int32)
    md, keep = h.metric._desc(D, N, z.theta)
    e, ep, keep2 = _eps_args(step_size(lf), z.theta, N)
    alpha = lf.alpha if isinstance(lf, TemperedLeapfrog) else 0.0
    host = _is_host(z.theta)
    _sync_torch(z.theta)
    zc, oc = z._c(), out._c(with_lk_gradient)
    ctx.check(ctx.lib.ahmc_leapfrog_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, int(n_steps), alpha,
                                        C.byref(zc), C.byref(oc), _ptr(status), _ptr(done),
                                        flags | (L.FLAG_HOST_BUFFERS if host else 0)))
    return (out, StepInfo(status, done)) if return_info else out


class StepPlan:
    """A prepared `step` call: buffers, descriptors and ctypes arguments are bound once, `plan()` then
    costs one foreign call (a few microseconds of host time) -- use it when the same shapes are stepped
    repeatedly (sampling loops, benchmarks).  `z` and `out` keep their identity; pass out=z for in place."""

    def __init__(self, lf: AbstractLeapfrog, h: Hamiltonian, z: PhasePoint, n_steps: int, out: Optional[PhasePoint] = None,
                 flags: int = 0, with_info: bool = False):
        self.ctx = ctx = get_context(_device_of(z.theta))
        N, D = z._nd()
        self.z, self.out = z, (out if out is not None else _empty_pp(z.theta, with_lk_gradient=False))
        self.status = _like(z.theta, (N,), np.uint32) if with_info else None
        self.steps_done = _like(z.theta, (N,), np.int32) if with_info else None
        self._md, self._keep = h.metric._desc(D, N, z.theta)
        e, ep, self._keep2 = _eps_args(step_size(lf), z.theta, N)
        alpha = lf.alpha if isinstance(lf, TemperedLeapfrog) else 0.0
        self._zc, self._oc = z._c(), self.out._c(self.out.lk.gradient is not None)
        fl = flags | (L.FLAG_HOST_BUFFERS if _is_host(z.theta) else 0)
        self._args = (ctx.h, h.target.handle(ctx), C.byref(self._md), D, N, e, ep, int(n_steps), alpha,
                      C.byref(self._zc), C.byref(self._oc), _ptr(self.status), _ptr(self.steps_done), fl)
        self._fn = ctx.lib.ahmc_leapfrog_f64
        self._h = h

    def __call__(self) -> PhasePoint:
        rc = self._fn(*self._args)
        if rc != L.OK:
            self.ctx.check(rc)
        return self.out


def _step_full_trajectory(lf, h, z, n_steps, flags):
    """`step(...; full_trajectory = Val(true))` (integrator.jl:229,249-261): returns (list of PhasePoint views,
    steps_done).  Like the reference's matrix mode the list has max(steps_done) entries; a chain that stopped
    early (per-chain break) leaves its later entries untouched -- consult steps_done."""
    ctx = get_context(_device_of(z.theta))
    N, D = z._nd()
    L_ = abs(n_steps)
    like = z.theta
    shp = (L_, N, D)
    traj = dict(theta=_like(like, shp), r=_like(like, shp), g=_like(like, shp), dr=_like(like, shp),
                lp=_like(like, (L_, N)), lk=_like(like, (L_, N)))
    done = _like(like, (N,), np.int32)
    if L_ == 0:
        return [], done
    md, keep = h.metric._desc(D, N, like)
    e, ep, keep2 = _eps_args(step_size(lf), like, N)
    alpha = lf.alpha if isinstance(lf, TemperedLeapfrog) else 0.0
    tc = L.PhasePoint(_ptr(traj["theta"]), _ptr(traj["r"]), _ptr(traj["lp"]), _ptr(traj["g"]), _ptr(traj["lk"]),
                      _ptr(traj["dr"]), D)
    _sync_torch(like)
    zc = z._c()
    ctx.check(ctx.lib.ahmc_leapfrog_trajectory_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, int(n_steps),
                                                   alpha, C.byref(zc), C.byref(tc), N * D, _ptr(done),
                                                   flags | (L.FLAG_HOST_BUFFERS if _is_host(like) else 0)))
    nmax = int(done.max()) if N else 0
    zs = [PhasePoint(traj["theta"][i], traj["r"][i], DualValue(traj["lp"][i], traj["g"][i]),
                     DualValue(traj["lk"][i], traj["dr"][i])) for i in range(nmax)]
    return zs, done


# ------------------------------------------------------------------------------------------------
# trajectories / kernels (src/trajectory.jl)
# ------------------------------------------------------------------------------------------------
class EndPointTS:
    pass


class MultinomialTS:
    pass


class SliceTS:
    """Slice trajectory sampler (trajectory.jl:102-109); dynamic trajectories only."""


@dataclass(frozen=True)
class FixedNSteps:
    L: int


@dataclass(frozen=True)
class FixedIntegrationTime:
    lam: float


@dataclass(frozen=True)
class GeneralisedNoUTurn:
    max_depth: int = 10
    delta_max: float = 1000.0


@dataclass(frozen=True)
class ClassicNoUTurn:
    """trajectory.jl:240-250, isterminated at :551-557."""
    max_depth: int = 10
    delta_max: float = 1000.0


@dataclass(frozen=True)
class StrictGeneralisedNoUTurn:
    """trajectory.jl:272-282, isterminated at :579-613."""
    max_depth: int = 10
    delta_max: float = 1000.0


_DYNAMIC = (GeneralisedNoUTurn, ClassicNoUTurn, StrictGeneralisedNoUTurn)


def _nuts_flags(tau):
    """Flag bits selecting the trajectory sampler / criterion of a dynamic trajectory."""
    if tau.sampler is MultinomialTS:
        fl = 0
    elif tau.sampler is SliceTS:
        fl = L.FLAG_NUTS_SLICE_TS
    else:
        raise L.AhmcError(L.ERR_UNSUPPORTED, "dynamic trajectories: MultinomialTS or SliceTS")
    tc = tau.termination_criterion
    if isinstance(tc, ClassicNoUTurn):
        fl |= L.FLAG_NUTS_CLASSIC
    elif isinstance(tc, StrictGeneralisedNoUTurn):
        fl |= L.FLAG_NUTS_STRICT
    return fl


@dataclass(frozen=True)
class Trajectory:
    """Trajectory{TS}(integrator, termination_criterion) (trajectory.jl:213-224)."""

    sampler: type
    integrator: AbstractIntegrator
    termination_criterion: Any


def nsteps(tau: Trajectory) -> int:
    """trajectory.jl:240-243."""
    tc = tau.termination_criterion
    if isinstance(tc, FixedNSteps):
        return tc.L
    eps = nom_step_size(tau.integrator)
    if np.ndim(eps) != 0:
        raise L.InvalidArgument(L.ERR_INVALID, "FixedIntegrationTime needs a scalar step size (quirk Q6, trajectory.jl:241-243)")
    return max(1, math.floor(tc.lam / eps))


class FullMomentumRefreshment:
    """src/hamiltonian.jl:210-220."""


@dataclass(frozen=True)
class PartialMomentumRefreshment:
    """src/hamiltonian.jl:222-254: r' = alpha*r + sqrt(1 - alpha^2)*G."""

    alpha: float


def _refresh_alpha(kappa) -> float:
    r = getattr(kappa, "refreshment", None)
    return float(r.alpha) if isinstance(r, PartialMomentumRefreshment) else 0.0


def _temper_alpha(lf) -> float:
    return float(lf.alpha) if isinstance(lf, TemperedLeapfrog) else 0.0


@dataclass(frozen=True)
class HMCKernel:
    """trajectory.jl:249-254."""

    tau: Trajectory
    refreshment: Any = field(default_factory=FullMomentumRefreshment)


@dataclass
class Transition:
    """trajectory.jl:18-23."""

    z: PhasePoint
    stat: dict


def _stats_buffers(like, N, nuts, T=None):
    shp = (N,) if T is None else (T, N)
    s = dict(n_steps=_like(like, shp, np.int32), is_accept=_like(like, shp, np.uint8),
             acceptance_rate=_like(like, shp), log_density=_like(like, shp), hamiltonian_energy=_like(like, shp),
             hamiltonian_energy_error=_like(like, shp), numerical_error=_like(like, shp, np.uint8))
    if nuts:
        s["max_hamiltonian_energy_error"] = _like(like, shp)
        s["tree_depth"] = _like(like, shp, np.int32)
    c = L.Stats(_ptr(s["n_steps"]), _ptr(s["is_accept"]), _ptr(s["acceptance_rate"]), _ptr(s["log_density"]),
                _ptr(s["hamiltonian_energy"]), _ptr(s["hamiltonian_energy_error"]),
                _ptr(s.get("max_hamiltonian_energy_error")), _ptr(s.get("tree_depth")), _ptr(s["numerical_error"]))
    return s, c


def _jitter_generator(rng) -> np.random.Generator:
    """host uniforms for `jitter` (integrator.jl:140-156), reproducible from the transition's rng"""
    if isinstance(rng, PhiloxRNG):
        return np.random.Generator(np.random.Philox(key=rng.seed, counter=[1, 0, 0, rng.offset]))
    if isinstance(rng, np.random.Generator):
        return rng
    g = getattr(rng, "_jitter_gen", None)
    if g is None:
        g = np.random.default_rng(0)
        try:
            rng._jitter_gen = g
        except Exception:
            pass
    return g


def transition(rng, h: Hamiltonian, kappa: Union[HMCKernel, Trajectory], z: PhasePoint, flags: int = 0) -> Transition:
    """`transition(rng, h, kappa, z)` (sampler.jl:48-58 -> trajectory.jl:271-300 static / :677-742 NUTS).
    With an HMCKernel the momentum is refreshed first; with a bare Trajectory z.r is used as is."""
    if isinstance(kappa, HMCKernel):
        tau = kappa.tau
    else:
        tau, flags = kappa, flags | L.FLAG_NO_REFRESH
    ctx = get_context(_device_of(z.theta))
    N, D = z._nd()
    host = _is_host(z.theta)
    out = _empty_pp(z.theta, with_lk_gradient=False)
    md, keep = h.metric._desc(D, N, z.theta)
    lf = tau.integrator
    if isinstance(lf, JitteredLeapfrog):
        # `@set! tau.integrator = jitter(rng, tau.integrator)` (src/sampler.jl, transition): a fresh jittered step size per
        # transition, derived from the nominal one (so a dual-averaging update of eps0 takes effect).  The jitter uniforms
        # come from a host generator keyed by the transition's own rng state.
        lf = jitter(_jitter_generator(rng), lf)
    e, ep, keep2 = _eps_args(step_size(lf), z.theta, N)
    rc, keep3 = rng._c()
    rc.partial_refresh_alpha = _refresh_alpha(kappa)
    rc.temper_alpha = _temper_alpha(lf)  # TemperedLeapfrog: every `step` of the transition tempers by its own n_steps
    tc = tau.termination_criterion
    nuts = isinstance(tc, _DYNAMIC)
    st, sc = _stats_buffers(z.theta, N, nuts or tau.sampler is MultinomialTS)
    fl = flags | (L.FLAG_HOST_BUFFERS if host else 0)
    _sync_torch(z.theta)
    zc, oc = z._c(False), out._c(False)
    if nuts:
        fl |= _nuts_flags(tau)
        ctx.check(ctx.lib.ahmc_nuts_transition_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep,
                                                   tc.max_depth, tc.delta_max, C.byref(rc), C.byref(zc),
                                                   C.byref(oc), C.byref(sc), fl))
    elif tau.sampler is MultinomialTS:
        # the direction split is ONE draw shared by all chains, like `rand_coupled(rng, 0:n_steps)` (trajectory.jl:371-373)
        n = nsteps(tau)
        n_fwd = rng.draw_n_fwd(n)
        ctx.check(ctx.lib.ahmc_hmc_multinomial_transition_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, n,
                                                              n_fwd, C.byref(rc), C.byref(zc), C.byref(oc),
                                                              C.byref(sc), fl))
        st["n_steps_fwd"] = n_fwd
    else:
        if tau.sampler is not EndPointTS:
            raise L.AhmcError(L.ERR_UNSUPPORTED, "static trajectories: EndPointTS or MultinomialTS")
        ctx.check(ctx.lib.ahmc_hmc_transition_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, nsteps(tau),
                                                  C.byref(rc), C.byref(zc), C.byref(oc), C.byref(sc), fl))
    st.update(stat(lf))
    return Transition(out, st)


def find_good_stepsize(rng, h: Hamiltonian, theta, initial_step_size: float = 0.1, max_n_iters: int = 100) -> float:
    """`find_good_stepsize(rng, h, theta)` (src/trajectory.jl:768-837): doubling / halving until the one-step
    acceptance ratio crosses 1/2, then bisection until it lies in (1/4, 3/4].  Host-side control flow exactly
    as the reference (it runs once); every probe `A(h, z, eps)` (:753-757) is one call of the fused `step` kernel.
    `theta`: one chain, shape (D,) (the reference accepts a vector only)."""
    if theta.ndim != 1:
        raise L.InvalidArgument(L.ERR_INVALID, "find_good_stepsize takes a single chain (vector theta), like the reference")
    th = theta.reshape(1, -1)
    r = rand_momentum(rng, h.metric, h.kinetic, th)
    z = phasepoint(h, th, r)
    H = float(energy(z)[0])

    def A_(eps):  # trajectory.jl:753-757
        z1 = step(Leapfrog(eps), h, z, 1, with_lk_gradient=False)
        return float(energy(z1)[0])

    eps = eps_prime = float(initial_step_size)
    log_a_min, log_a_cross, log_a_max = 2 * math.log(0.5), math.log(0.5), math.log(0.75)
    dH = H - A_(eps)
    ratio_too_high = dH > log_a_cross
    for _ in range(max_n_iters):  # crossing step (:796-810)
        eps_prime = 2.0 * eps if ratio_too_high else 0.5 * eps
        dH = H - A_(eps)
        if ratio_too_high != (dH > log_a_cross):
            break
        eps = eps_prime
    eps, eps_prime = min(eps, eps_prime), max(eps, eps_prime)
    for _ in range(max_n_iters):  # bisection (:822-834)
        mid = 0.5 * (eps + eps_prime)
        dH = H - A_(mid)
        if dH > log_a_max:
            eps = mid
        elif dH < log_a_min:
            eps_prime = mid
        else:
            eps = mid
            break
    return eps


def find_good_stepsize_batched(rng, h: Hamiltonian, theta, initial_step_size: float = 0.1, max_n_iters: int = 100,
                               return_momentum: bool = False):
    """N independent copies of `find_good_stepsize` (src/trajectory.jl:768-837), one per chain of `theta` (N, D), in ONE
    kernel launch (ahmc_find_good_stepsize_f64): momentum draw, direction probe, crossing loop and bisection all run on the
    device, each chain at its own pace -- no host round trip.  Returns eps (N,) -- the natural starting point for the
    vectorised adaptors (`VectorisedStanAdaptor`).  Chain c's result equals `find_good_stepsize` on that chain alone with
    the same momentum."""
    if theta.ndim != 2:
        raise L.InvalidArgument(L.ERR_INVALID, "find_good_stepsize_batched takes (N, D) positions")
    N, D = theta.shape
    ctx = get_context(_device_of(theta))
    z = phasepoint(h, theta, _like(theta, (N, D)) * 0 if _is_host(theta) else torch.zeros_like(theta))
    md, keep = h.metric._desc(D, N, theta)
    rc, keep2 = rng._c()
    eps = _like(theta, (N,))
    r = _like(theta, (N, D)) if return_momentum else None
    _sync_torch(theta)
    zc = z._c(False)
    ctx.check(ctx.lib.ahmc_find_good_stepsize_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, C.byref(zc), C.byref(rc),
                                                  float(initial_step_size), int(max_n_iters), _ptr(eps), _ptr(r),
                                                  L.FLAG_HOST_BUFFERS if _is_host(theta) else 0))
    return (eps, r) if return_momentum else eps


def sample_transitions(rng: PhiloxRNG, h: Hamiltonian, kappa: HMCKernel, z: PhasePoint, n_transitions: int,
                       keep_draws: bool = True, flags: int = 0):
    """`n_transitions` consecutive transitions per chain in ONE kernel launch -- the un-adapted body of
    `sample` (src/sampler.jl:182-228): returns (z_last, draws (T, N, D) or None, stats dict of (T, N) arrays).
    Chains advance at their own pace inside the launch (no barrier between transitions)."""
    if not isinstance(rng, PhiloxRNG):
        raise L.InvalidArgument(L.ERR_INVALID, "multi-transition sampling draws from the on-device Philox streams")
    tau = kappa.tau
    ctx = get_context(_device_of(z.theta))
    N, D = z._nd()
    host = _is_host(z.theta)
    out = _empty_pp(z.theta, with_lk_gradient=False)
    md, keep = h.metric._desc(D, N, z.theta)
    lf = tau.integrator
    if type(lf) not in (Leapfrog, TemperedLeapfrog):
        raise L.AhmcError(L.ERR_UNSUPPORTED, "multi-transition launches run Leapfrog / TemperedLeapfrog (a JitteredLeapfrog draws a new "
                                              "step size per transition on the host): loop over transition()")
    tc = tau.termination_criterion
    nuts = isinstance(tc, _DYNAMIC)
    if not nuts and tau.sampler is not EndPointTS:
        raise L.AhmcError(L.ERR_UNSUPPORTED, "multi-transition static launches implement EndPointTS (Metropolis end point); a static "
                                              "MultinomialTS trajectory needs one shared direction draw per transition: loop over transition()")
    e, ep, keep2 = _eps_args(step_size(lf), z.theta, N)
    rc = L.Rng(rng.seed, rng.offset, None, None, 0, None, 0, _refresh_alpha(kappa), _temper_alpha(kappa.tau.integrator))
    rng.offset += n_transitions
    st, sc = _stats_buffers(z.theta, N, nuts, T=n_transitions)
    draws = _like(z.theta, (n_transitions, N, D)) if keep_draws else None
    fl = flags | (L.FLAG_HOST_BUFFERS if host else 0)
    _sync_torch(z.theta)
    zc, oc = z._c(False), out._c(False)
    if nuts:
        fl |= _nuts_flags(tau)
        ctx.check(ctx.lib.ahmc_nuts_sample_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, tc.max_depth,
                                               tc.delta_max, n_transitions, C.byref(rc), C.byref(zc), C.byref(oc),
                                               _ptr(draws), C.byref(sc), fl))
    else:
        ctx.check(ctx.lib.ahmc_hmc_sample_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, e, ep, nsteps(tau),
                                              n_transitions, C.byref(rc), C.byref(zc), C.byref(oc), _ptr(draws),
                                              C.byref(sc), fl))
    st.update(stat(lf))
    return out, draws, st


@dataclass
class VectorisedStanAdaptor:
    """`StanHMCAdaptor(WelfordVar((D, N)), NesterovDualAveraging(delta, eps::Vector))`: the reference's vectorised
    adaptors -- one dual-averaging state and one windowed variance estimator PER CHAIN (stepsize.jl:178-210,
    massmatrix.jl:141-157, stan_adaptor.jl:13-50, 137-159).  Runs inside the NUTS launch (ahmc_nuts_adapt_sample_f64)."""
    delta: float = 0.8
    adapt_metric: bool = True
    init_buffer: int = 75
    term_buffer: int = 50
    window_size: int = 25
    gamma: float = 0.05
    t0: float = 10.0
    kappa: float = 0.75
    n_min: int = 10


def nuts_adapt_sample(rng: PhiloxRNG, h: Hamiltonian, kappa: HMCKernel, z: PhasePoint, n_transitions: int, n_adapts: int,
                      adaptor: VectorisedStanAdaptor, keep_draws: bool = True, keep_eps_trace: bool = False, flags: int = 0):
    """n_adapts adapting + (n_transitions - n_adapts) sampling NUTS transitions per chain in ONE launch, every chain
    adapting its own step size (and diagonal metric).  -> (z_last, draws (T, N, D) | None, stats of (T, N) arrays,
    eps (N,), Minv (N, D) | None, eps_trace (T, N) | None).  The initial step size is `step_size(kappa.tau.integrator)`
    (scalar or per chain), the initial metric h.metric (DiagEuclideanMetric)."""
    if not isinstance(rng, PhiloxRNG):
        raise L.InvalidArgument(L.ERR_INVALID, "in-launch adaptation draws from the on-device Philox streams")
    tau = kappa.tau
    if tau.sampler is not MultinomialTS or not isinstance(tau.termination_criterion, GeneralisedNoUTurn):
        raise L.AhmcError(L.ERR_UNSUPPORTED, "in-launch adaptation: MultinomialTS + GeneralisedNoUTurn")
    ctx = get_context(_device_of(z.theta))
    N, D = z._nd()
    host = _is_host(z.theta)
    out = _empty_pp(z.theta, with_lk_gradient=False)
    md, keep = h.metric._desc(D, N, z.theta)
    e0 = step_size(tau.integrator)
    eps = _like(z.theta, (N,))
    if np.ndim(e0) == 0:
        eps[...] = float(e0)
    elif host:
        eps[...] = np.asarray(e0, dtype=np.float64)
    else:
        eps.copy_(e0 if hasattr(e0, "detach") else torch.as_tensor(np.asarray(e0, dtype=np.float64)))
    minv = _like(z.theta, (N, D)) if adaptor.adapt_metric else None
    trace = _like(z.theta, (n_transitions, N)) if keep_eps_trace else None
    cfg = L.AdaptCfg(n_adapts, adaptor.init_buffer, adaptor.term_buffer, adaptor.window_size, adaptor.delta, adaptor.gamma,
                     adaptor.t0, adaptor.kappa, 1 if adaptor.adapt_metric else 0, adaptor.n_min, _ptr(eps), _ptr(minv),
                     _ptr(trace))
    rc = L.Rng(rng.seed, rng.offset, None, None, 0, None, 0, _refresh_alpha(kappa), _temper_alpha(kappa.tau.integrator))
    rng.offset += n_transitions
    tc = tau.termination_criterion
    st, sc = _stats_buffers(z.theta, N, True, T=n_transitions)
    draws = _like(z.theta, (n_transitions, N, D)) if keep_draws else None
    fl = flags | (L.FLAG_HOST_BUFFERS if host else 0)
    _sync_torch(z.theta)
    zc, oc = z._c(False), out._c(False)
    ctx.check(ctx.lib.ahmc_nuts_adapt_sample_f64(ctx.h, h.target.handle(ctx), C.byref(md), D, N, tc.max_depth, tc.delta_max,
                                                 n_transitions, C.byref(cfg), C.byref(rc), C.byref(zc), C.byref(oc),
                                                 _ptr(draws), C.byref(sc), fl))
    return out, draws, st, eps, minv, trace


# ------------------------------------------------------------------------------------------------
# adaptor statistics (src/adaptation): pooled summary record of one iteration
# ------------------------------------------------------------------------------------------------
def adapt_summary(theta, acceptance_rate):
    """-> float64 array [N, sum min(1,alpha), mean[D], M2[D]] (device tensor or numpy), see ahmc_adapt_summary_f64."""
    ctx = get_context(_device_of(theta))
    N, D = tuple(theta.shape)
    out = _like(theta, (2 + 2 * D,))
    _sync_torch(theta)
    ctx.check(ctx.lib.ahmc_adapt_summary_f64(ctx.h, D, N, _ptr(theta), D, _ptr(acceptance_rate), _ptr(out),
                                             L.FLAG_HOST_BUFFERS if _is_host(theta) else 0))
    return out


def adapt_cov(theta, mean):
    """-> (D, D) float64 second-moment matrix sum_c (theta_c - mean)(theta_c - mean)' (ahmc_adapt_cov_f64);
    `mean` = adapt_summary(theta, .)[2:2+D]."""
    ctx = get_context(_device_of(theta))
    N, D = tuple(theta.shape)
    out = _like(theta, (D, D))
    _sync_torch(theta)
    ctx.check(ctx.lib.ahmc_adapt_cov_f64(ctx.h, D, N, _ptr(theta), D, _ptr(mean), _ptr(out),
                                         L.FLAG_HOST_BUFFERS if _is_host(theta) else 0))
    return out


# ------------------------------------------------------------------------------------------------
# deployment helper: host-buffer calls move every byte over PCIe, so the page-locked buffers should live on the NUMA
# node the GPU hangs off (on a two-socket B200 box a remote node costs up to ~1.5x per call, profiles/README.md)
# ------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(device: int = 0):
    """Pin the calling thread to the CPUs NVML reports as local to `device` (nvmlDeviceSetCpuAffinity) so that memory
    it allocates and first-touches afterwards -- e.g. `torch.Tensor.pin_memory()` buffers handed to the
    AHMC_FLAG_HOST_BUFFERS calls -- lands on the GPU's NUMA node.  Returns the previous affinity set (pass it to
    `os.sched_setaffinity(0, prev)` to undo) or None when NVML / the cpuset does not allow it."""
    import os

    try:
        import pynvml

        pynvml.nvmlInit()
        handle = None
        try:
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid if not uuid.startswith("GPU-") else uuid).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(device)
        prev = os.sched_getaffinity(0)
        pynvml.nvmlDeviceSetCpuAffinity(handle)
        return prev
    except Exception:
        return None
