"""Torch-facing operators over the C ABI (include/mcpilco_b200.h).

PyTorch supplies device memory, the current stream and autograd bookkeeping; all arithmetic of the hot
path runs in libmcpilco_b200.so.  Every function here rejects non-CUDA / non-float64 tensors: there is
no CPU fallback and no alternative backend.
"""
import ctypes as C

import torch

from . import _native as N
from . import _pack as P

F64 = torch.float64


_ws_cache = {}


def _need_cuda(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != F64:
        raise RuntimeError("mcpilco_b200: %s must be a CUDA float64 tensor (this path has no CPU fallback); got %s"
                           % (name, "%s/%s" % (t.device, t.dtype) if isinstance(t, torch.Tensor) else type(t)))
    return t


def _c(t, name):
    return _need_cuda(t, name).detach().contiguous()


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _enter(dev):
    L = N.lib()
    N.check(L.mcpilco_set_device(dev.index if dev.index is not None else torch.cuda.current_device()))
    return L


def _restores_device(fn):
    """The native entry points make the tensors' device current (kernel launches need it); put the caller's device back afterwards so
    that an op on cuda:1 does not silently redirect the caller's later `device="cuda"` allocations."""
    import functools

    @functools.wraps(fn)
    def wrapped(*a, **k):
        prev = torch.cuda.current_device() if torch.cuda.is_available() else None
        try:
            return fn(*a, **k)
        finally:
            if prev is not None and torch.cuda.current_device() != prev:
                N.lib().mcpilco_set_device(prev)
    return wrapped


def even_ld(n):
    return n + (n & 1)


# ---------------------------------------------------------------------------------------------------
# covariance / precompute / posterior
# ---------------------------------------------------------------------------------------------------
@_restores_device
def gp_covariance(spec, X1, X2=None, add_noise=False):
    """k(X1, X2) [+ sigma_n2 I].  GP_prior.py:314-335 and children."""
    X1 = _c(X1, "X1")
    L = _enter(X1.device)
    if X1.dim() != 2 or X1.shape[1] != spec.D:
        raise RuntimeError("gp_covariance: X1 must be [n, %d]" % spec.D)
    n1 = X1.shape[0]
    if X2 is not None:
        X2 = _c(X2, "X2")
        if X2.dim() != 2 or X2.shape[1] != spec.D:
            raise RuntimeError("gp_covariance: X2 must be [n, %d]" % spec.D)
    n2 = n1 if X2 is None else X2.shape[0]
    K = torch.empty(n1, n2, dtype=F64, device=X1.device)
    if n1 and n2:
        N.check(L.mcpilco_gp_covariance(C.byref(spec), _ptr(X1), n1, _ptr(X2), n2, 1 if add_noise else 0, _ptr(K), n2,
                                        _stream(X1.device)))
    return K


@_restores_device
def gp_diag_covariance(spec, X):
    """diag k(X, X) without noise.  GP_prior.py:337-347."""
    X = _c(X, "X")
    L = _enter(X.device)
    out = torch.empty(X.shape[0], dtype=F64, device=X.device)
    if X.shape[0]:
        N.check(L.mcpilco_gp_diag_covariance(C.byref(spec), _ptr(X), X.shape[0], _ptr(out), _stream(X.device)))
    return out


@_restores_device
def gp_precompute(spec, Xtr, y, want_L=False, want_Linv=False):
    """alpha [N,1], K^-1 [N,N] (a view of an [N, even_ld(N)] buffer, as the posterior kernels want it) and optionally the
    Cholesky factor L and / or its inverse R = L^-1 (lower triangular; what forward-only posteriors contract with).
    GP_prior.py:91-115,130-135."""
    Xtr, y = _c(Xtr, "X"), _c(y, "Y").reshape(-1)
    L_ = _enter(Xtr.device)
    n = Xtr.shape[0]
    if n < 1 or Xtr.shape[1] != spec.D or y.numel() != n:
        raise RuntimeError("gp_precompute: X must be [N>=1, %d] and Y [N, 1]" % spec.D)
    ld = even_ld(n)
    alpha = torch.empty(n, dtype=F64, device=Xtr.device)
    Kbuf = torch.zeros(n, ld, dtype=F64, device=Xtr.device)
    Lbuf = torch.zeros(n, ld, dtype=F64, device=Xtr.device) if want_L else None
    Rbuf = torch.zeros(n, ld, dtype=F64, device=Xtr.device) if want_Linv else None
    wsb = L_.mcpilco_gp_precompute_workspace_bytes(n)
    ws = torch.empty(wsb, dtype=torch.uint8, device=Xtr.device)
    N.check(L_.mcpilco_gp_precompute(C.byref(spec), _ptr(Xtr), _ptr(y), n, _ptr(alpha), _ptr(Kbuf), ld, _ptr(Lbuf), _ptr(Rbuf), _ptr(ws), wsb,
                                     _stream(Xtr.device)))
    out = (alpha.reshape(n, 1), Kbuf[:, :n])
    if want_L:
        out = out + (Lbuf[:, :n],)
    if want_Linv:
        out = out + (Rbuf[:, :n],)
    return out


@_restores_device
def gp_nlml(spec, Xtr, y):
    """Negative marginal log likelihood and its gradient w.r.t. the McpGpSpec fields, as one device tensor (layout:
    include/mcpilco_b200.h, mcpilco_gp_nlml).  GP_prior.py:91-115,179-230; Gaussian_likelihood.py:12-24."""
    Xtr, y = _c(Xtr, "X"), _c(y, "Y").reshape(-1)
    L_ = _enter(Xtr.device)
    n = Xtr.shape[0]
    if n < 1 or Xtr.shape[1] != spec.D or y.numel() != n:
        raise RuntimeError("gp_nlml: X must be [N>=1, %d] and Y [N, 1]" % spec.D)
    out = torch.empty(L_.mcpilco_gp_nlml_grad_size(), dtype=F64, device=Xtr.device)
    wsb = L_.mcpilco_gp_nlml_workspace_bytes(n)
    ws = _workspace(Xtr.device, wsb, "nlml")
    N.check(L_.mcpilco_gp_nlml(C.byref(spec), _ptr(Xtr), _ptr(y), n, _ptr(out), _ptr(ws), ws.numel(), _stream(Xtr.device)))
    return out


@_restores_device
def gp_sod_select(spec, X, threshold, order=None):
    """Greedy subset-of-data selection on the device; returns the selected indices (python list, in selection order).
    GP_prior.py:232-257."""
    X = _c(X, "X")
    L_ = _enter(X.device)
    n = X.shape[0]
    if n < 1 or X.shape[1] != spec.D:
        raise RuntimeError("gp_sod_select: X must be [N>=1, %d]" % spec.D)
    idx = torch.empty(n, dtype=torch.int32, device=X.device)
    cnt = torch.zeros(1, dtype=torch.int32, device=X.device)
    od = None if order is None else torch.as_tensor(order, dtype=torch.int32, device=X.device).contiguous()
    wsb = L_.mcpilco_gp_sod_workspace_bytes(n)
    ws = _workspace(X.device, wsb, "sod")
    N.check(L_.mcpilco_gp_sod_select(C.byref(spec), _ptr(X), n, _ptr(od), float(threshold), _ptr(idx), _ptr(cnt), _ptr(ws), ws.numel(),
                                     _stream(X.device)))
    k = int(cnt.item())
    return [int(i) for i in idx[:k].tolist()]


NLML_LAMBDA, NLML_MEAN, NLML_SN2, NLML_ILS = 1, 2, 3, 4


def nlml_poly_offset(p, f):
    return 4 + N.MAX_D + (p * N.MAX_DEG + f) * (N.MAX_D + 1)


def kinv_for_kernels(Kinv):
    """Return (tensor, ld) with a 16-byte aligned base and an even leading dimension; copies only if needed."""
    _need_cuda(Kinv, "K_X_inv")
    n = Kinv.shape[0]
    if Kinv.dim() != 2 or Kinv.shape[1] != n:
        raise RuntimeError("K_X_inv must be square")
    if Kinv.stride(1) == 1 and Kinv.stride(0) >= n and Kinv.stride(0) % 2 == 0 and Kinv.data_ptr() % 16 == 0:
        return Kinv, Kinv.stride(0)
    buf = torch.zeros(n, even_ld(n), dtype=F64, device=Kinv.device)
    buf[:, :n].copy_(Kinv.detach())
    return buf[:, :n], buf.stride(0)


def attach_linv(Kinv, Linv):
    """Remember the triangular factor L^-1 that belongs to this K^-1 tensor (valid while the tensor is not modified in place)."""
    Kinv._mcp_linv = (Linv, Kinv._version, Kinv.data_ptr())


def attached_linv(Kinv):
    tag = getattr(Kinv, "_mcp_linv", None)
    if tag is None or tag[1] != Kinv._version or tag[2] != Kinv.data_ptr():
        return None
    return tag[0]


class FittedGp:
    """One output's fitted GP: what Model_learning keeps per gp_index (Model_learning.py:172-175)."""

    @_restores_device
    def __init__(self, spec, Xtr, alpha, Kinv, var_scale=1.0, ozaki_slices=None, Linv=None):
        """ozaki_slices: None -> environment MCPILCO_OZAKI (default 0 = native FP64 contraction); 7 or 8 -> the opt-in INT8
        tensor-core contraction with error compensation (include/mcpilco_b200.h, mcpilco_ozaki_prepare)."""
        self.spec = spec
        self.Xtr = _c(Xtr, "gp_inputs")
        self.alpha = _c(alpha, "alpha").reshape(-1)
        self.Kinv, self.ld = kinv_for_kernels(Kinv)
        # optional triangular factor L^-1 (gp_precompute(want_Linv=True)): forward-only posteriors / rollouts then cost N^2 flops
        if Linv is None:
            Linv = attached_linv(Kinv)
        self.Linv, self.ld_linv = kinv_for_kernels(Linv) if Linv is not None else (None, 0)
        if self.Linv is not None and self.Linv.shape[0] != self.Kinv.shape[0]:
            raise RuntimeError("FittedGp: Linv and Kinv sizes differ")
        self.var_scale = float(var_scale)
        self.N = self.Xtr.shape[0]
        if self.Xtr.shape[1] != spec.D or self.alpha.numel() != self.N or self.Kinv.shape[0] != self.N:
            raise RuntimeError("FittedGp: inconsistent shapes")
        import os
        self.ozaki = int(os.environ.get("MCPILCO_OZAKI", "0")) if ozaki_slices is None else int(ozaki_slices)
        self.planes = self.plane_exp = None
        self.kdiag_max = 0.0
        if self.ozaki:
            L = _enter(self.Xtr.device)
            if not L.mcpilco_ozaki_available():
                raise RuntimeError("mcpilco_b200: the INT8 (Ozaki) contraction was requested but this build has no CUTLASS headers")
            if self.ozaki not in (7, 8):
                raise RuntimeError("mcpilco_b200: ozaki_slices must be 7 or 8")
            self.planes = torch.empty(L.mcpilco_ozaki_plane_bytes(self.N, self.ozaki), dtype=torch.uint8, device=self.Xtr.device)
            self.plane_exp = torch.empty(self.N, dtype=torch.int32, device=self.Xtr.device)
            N.check(L.mcpilco_ozaki_prepare(_ptr(self.Kinv), self.N, self.ld, self.ozaki, _ptr(self.planes), _ptr(self.plane_exp),
                                            _stream(self.Xtr.device)))
            # bound for the rows of K* (Cauchy-Schwarz): lets the K* kernel choose the row scale and emit the digit planes itself
            kd = gp_diag_covariance(spec, self.Xtr).max()
            self.kdiag_max = float(kd) if bool(torch.isfinite(kd)) else 0.0

    @classmethod
    def from_parts(cls, spec, Xtr, alpha, Kinv, ld, var_scale, ozaki, planes, plane_exp, Linv, ld_linv, kdiag_max):
        """Re-assemble a FittedGp from tensors that already passed __init__ (the torch.library op layer ships them as flat arguments);
        no validation, no copies, no re-slicing of K^-1."""
        g = cls.__new__(cls)
        g.spec, g.Xtr, g.alpha, g.Kinv, g.ld, g.var_scale, g.N = spec, Xtr, alpha, Kinv, int(ld), float(var_scale), Xtr.shape[0]
        g.ozaki, g.planes, g.plane_exp, g.Linv, g.ld_linv, g.kdiag_max = int(ozaki), planes, plane_exp, Linv, int(ld_linv), float(kdiag_max)
        return g

    def fill(self, g):
        C.memmove(C.byref(g.spec), C.byref(self.spec), C.sizeof(N.GpSpec))
        g.N, g.ld_kinv = self.N, self.ld
        g.Xtr, g.alpha, g.Kinv = self.Xtr.data_ptr(), self.alpha.data_ptr(), self.Kinv.data_ptr()
        g.var_scale = self.var_scale
        g.ozaki_slices = self.ozaki
        g.kinv_planes = self.planes.data_ptr() if self.planes is not None else None
        g.kinv_exp = self.plane_exp.data_ptr() if self.plane_exp is not None else None
        g.Linv, g.ld_linv = (self.Linv.data_ptr(), self.ld_linv) if self.Linv is not None else (None, 0)
        g.kdiag_max = self.kdiag_max


def _gp_array(gps):
    arr = (N.Gp * len(gps))()
    for i, g in enumerate(gps):
        g.fill(arr[i])
    return arr


def _workspace(dev, nbytes, tag):
    """Grow-only scratch per (device, stream, tag): avoids a cudaMalloc round trip on every step."""
    key = (dev.index, torch.cuda.current_stream(dev).cuda_stream, tag)  # per stream: two streams never share scratch
    t = _ws_cache.get(key)
    if t is None or t.numel() < nbytes:
        t = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        _ws_cache[key] = t
    return t


def gp_predict(gps, Xs, jac=False):
    """Posterior mean/var [M, E] (and Jacobians [M, E, D]) of E fitted GPs at Xs.  GP_prior.py:137-155.

    Differentiable w.r.t. Xs (once): when grad mode is on and Xs requires grad, the forward takes the Jacobian path and the backward
    is  dL/dXs[m] = sum_e dL/dmean[m,e] jmean[m,e] + dL/dvar[m,e] jvar[m,e].  The fitted GPs (alpha, K^-1, training inputs, kernel
    parameters) receive no gradient.  Otherwise (and for jac=True) nothing is recorded and the outputs carry no graph."""
    if not jac and torch.is_grad_enabled() and isinstance(Xs, torch.Tensor) and Xs.requires_grad:
        return _GpPredict.apply(Xs, gps)
    return _gp_predict(gps, Xs, jac)


def gp_predict_vjp(jm, jv, g_mean, g_var):
    """dL/dXs [M, D] from the posterior Jacobians [M, E, D] and dL/dmean, dL/dvar [M, E] (either may be None)."""
    g = torch.zeros(jm.shape[0], jm.shape[2], dtype=F64, device=jm.device)
    if g_mean is not None:
        g = g + torch.einsum("me,med->md", g_mean, jm)
    if g_var is not None:
        g = g + torch.einsum("me,med->md", g_var, jv)
    return g


class _GpPredict(torch.autograd.Function):
    @staticmethod
    def forward(ctx, Xs, gps):
        mean, var, jm, jv = _gp_predict(gps, Xs, jac=True)
        ctx.save_for_backward(jm, jv)
        return mean, var

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_mean, g_var):
        jm, jv = ctx.saved_tensors
        return gp_predict_vjp(jm, jv, g_mean, g_var), None


@_restores_device
def _gp_predict(gps, Xs, jac=False):
    Xs = _c(Xs, "X_test")
    L = _enter(Xs.device)
    E, M, D = len(gps), Xs.shape[0], gps[0].spec.D
    if Xs.dim() != 2 or Xs.shape[1] != D:
        raise RuntimeError("gp_predict: X_test must be [M, %d]" % D)
    mean = torch.empty(M, E, dtype=F64, device=Xs.device)
    var = torch.empty(M, E, dtype=F64, device=Xs.device)
    jm = torch.empty(M, E, D, dtype=F64, device=Xs.device) if jac else None
    jv = torch.empty(M, E, D, dtype=F64, device=Xs.device) if jac else None
    if M:
        wsb = L.mcpilco_gp_predict_workspace_bytes(M, max(g.N for g in gps))
        ws = _workspace(Xs.device, wsb, "predict")
        arr = _gp_array(gps)
        N.check(L.mcpilco_gp_predict(arr, E, _ptr(Xs), M, _ptr(mean), _ptr(var), _ptr(jm), _ptr(jv), _ptr(ws), ws.numel(),
                                     _stream(Xs.device)))
    return (mean, var, jm, jv) if jac else (mean, var)


# ---------------------------------------------------------------------------------------------------
# rollout
# ---------------------------------------------------------------------------------------------------
class RolloutPlan:
    """Everything one rollout needs, flattened: owns the McpRollout struct and keeps every tensor it points to alive."""

    @_restores_device
    def __init__(self, model, gps, policy, pol_tensors, cost=None, cost_traj=None, meas=None, M=1, H=1, p_dropout=0.0,
                 seed=0, particle_offset=0, need_grad=False, eps=None, masks=None, meas_eps=None, device=None, M_global=0, seed_dev=None,
                 buffers=None):
        """buffers: optional {"states", "inputs", "jac", "pol_in"} of an earlier forward pass to adopt instead of allocating (the
        backward op of the torch.library layer rebuilds a plan around the trajectories autograd saved)."""
        self.dev = device or gps[0].Xtr.device
        self.L = _enter(self.dev)
        self.gps = list(gps)
        self.model, self.policy = model, policy
        self.cost = cost if cost is not None else N.Cost()
        self.meas = meas if meas is not None else N.Meas()
        self.M, self.H = int(M), int(H)
        self.need_grad = bool(need_grad)
        E, D, Ds, Du = model.E, model.D, model.Ds, model.Du
        if len(gps) != E:
            raise RuntimeError("rollout: %d fitted GPs for a model with %d outputs" % (len(gps), E))
        # policy tensors (device pointers are re-read at launch, so in-place optimiser updates are seen)
        self.log_ls, self.centers, self.W = (_need_cuda(pol_tensors[k], k) for k in ("log_ls", "centers", "W"))
        self.bias = _need_cuda(pol_tensors["bias"], "bias") if pol_tensors.get("bias") is not None else None
        self.traj = _c(pol_tensors["target_traj"], "target_traj") if pol_tensors.get("target_traj") is not None else None
        self.cost_traj = _c(cost_traj, "cost target_traj") if cost_traj is not None else None
        for t, nm in ((self.traj, "policy target_traj"), (self.cost_traj, "cost target_traj")):
            if t is not None and (t.dim() != 2 or t.shape[0] < H or t.shape[1] != Ds):
                raise RuntimeError("rollout: %s must be [>=H, Ds]" % nm)
        self.eps = _c(eps, "eps") if eps is not None else None
        self.masks = masks.detach().to(torch.uint8).contiguous() if masks is not None else None
        self.meas_eps = _c(meas_eps, "meas_eps") if meas_eps is not None else None
        if self.eps is not None and tuple(self.eps.shape) != (max(H - 1, 0), M, E):
            raise RuntimeError("rollout: eps must be [H-1, M, E]")
        if self.masks is not None and (not self.masks.is_cuda or tuple(self.masks.shape) != (H, M, policy.nb)):
            raise RuntimeError("rollout: masks must be a CUDA tensor [H, M, nb]")
        dev = self.dev
        bf = buffers or {}

        def buf(name, shape):
            t = bf.get(name)
            if t is None:
                return torch.empty(*shape, dtype=F64, device=dev)
            if tuple(t.shape) != tuple(shape) or not t.is_contiguous():
                raise RuntimeError("rollout: adopted buffer %s must be contiguous %s, got %s" % (name, tuple(shape), tuple(t.shape)))
            return _need_cuda(t, name)

        self.states = buf("states", (H, M, Ds))
        self.inputs = buf("inputs", (H, M, Du))
        self.jac = buf("jac", (max(H - 1, 1), M, E, D)) if need_grad else None
        self.pol_in = buf("pol_in", (H, M, Ds)) if self.meas.enabled else None
        fused = self.cost.kind != 0
        self.costs = torch.empty(H, M, dtype=F64, device=dev) if fused else None
        self.cost_out = torch.empty(2, dtype=F64, device=dev) if fused else None
        self.cost_stats = torch.empty(H, 2, dtype=F64, device=dev) if fused else None
        wsb = self.L.mcpilco_rollout_workspace_bytes(M, H, E, D, max(g.N for g in gps), policy.nb, policy.Dp, Du)
        self.ws = _workspace(dev, wsb, "rollout")
        self.gp_arr = _gp_array(self.gps)
        r = N.Rollout()
        r.M, r.H, r.need_grad, r.M_global = self.M, self.H, 1 if need_grad else 0, int(M_global)
        r.model, r.policy, r.cost, r.meas = model, policy, self.cost, self.meas
        r.noise.seed, r.noise.particle_offset, r.noise.p_dropout = int(seed), int(particle_offset), float(p_dropout)
        self.seed_dev = seed_dev  # optional device int64/uint64 word added to the seed at run time (graph replays)
        r.noise.seed_dev = seed_dev.data_ptr() if seed_dev is not None else None
        r.noise.eps = self.eps.data_ptr() if self.eps is not None else None
        r.noise.masks = self.masks.data_ptr() if self.masks is not None else None
        r.noise.meas_eps = self.meas_eps.data_ptr() if self.meas_eps is not None else None
        r.gps = C.cast(self.gp_arr, C.POINTER(N.Gp))
        for nm in ("states", "inputs", "jac", "pol_in", "costs", "cost_out", "cost_stats"):
            t = getattr(self, nm)
            setattr(r, nm, t.data_ptr() if t is not None else None)
        r.workspace, r.workspace_bytes = self.ws.data_ptr(), self.ws.numel()
        self.r = r
        self.x0 = None

    def _bind_policy(self):
        p = self.r.policy
        p.log_ls, p.centers, p.W = self.log_ls.data_ptr(), self.centers.data_ptr(), self.W.data_ptr()
        p.bias = self.bias.data_ptr() if self.bias is not None else None
        p.target_traj = self.traj.data_ptr() if self.traj is not None else None
        self.r.cost.target_traj = self.cost_traj.data_ptr() if self.cost_traj is not None else None
        for t, nm in ((self.log_ls, "log_lengthscales"), (self.centers, "centers"), (self.W, "weight")):
            if not t.is_contiguous():
                raise RuntimeError("rollout: policy tensor %s must be contiguous" % nm)

    @_restores_device
    def forward(self, x0):
        self.x0 = _c(x0, "x0")
        if tuple(self.x0.shape) != (self.M, self.model.Ds):
            raise RuntimeError("rollout: x0 must be [M, Ds]")
        self.r.x0 = self.x0.data_ptr()
        self._bind_policy()
        N.check(self.L.mcpilco_rollout_fwd(C.byref(self.r), _stream(self.dev)))
        return self.states, self.inputs

    @_restores_device
    def backward(self, grad_cost=0.0, grad_states=None, grad_inputs=None, want_gx0=False):
        """Policy-parameter gradients (flat views) of  grad_cost * expected_cost + <grad_states, states> + <grad_inputs, inputs>."""
        if not self.need_grad:
            raise RuntimeError("rollout backward: the forward pass was run without need_grad")
        pol = self.r.policy
        dev = self.dev
        g = N.RolloutGrad()
        gs = _c(grad_states, "grad_states") if grad_states is not None else None
        gi = _c(grad_inputs, "grad_inputs") if grad_inputs is not None else None
        out = {"log_ls": torch.empty(1, pol.Dp, dtype=F64, device=dev), "centers": torch.empty(pol.nb, pol.Dp, dtype=F64, device=dev),
               "W": torch.empty(pol.Du, pol.nb, dtype=F64, device=dev),
               "bias": torch.empty(pol.Du, dtype=F64, device=dev) if pol.has_bias else None,
               "x0": torch.empty(self.M, self.model.Ds, dtype=F64, device=dev) if want_gx0 else None}
        g.grad_states, g.grad_inputs, g.grad_cost = (gs.data_ptr() if gs is not None else None,
                                                     gi.data_ptr() if gi is not None else None, float(grad_cost))
        g.g_log_ls, g.g_centers, g.g_W = out["log_ls"].data_ptr(), out["centers"].data_ptr(), out["W"].data_ptr()
        g.g_bias = out["bias"].data_ptr() if out["bias"] is not None else None
        g.g_x0 = out["x0"].data_ptr() if out["x0"] is not None else None
        self._bind_policy()
        N.check(self.L.mcpilco_rollout_bwd(C.byref(self.r), C.byref(g), _stream(dev)))
        return out


def launch_count(reset=False):
    return int(N.lib().mcpilco_launch_count(1 if reset else 0))


def _policy_call_args(pst, tens, x, t, masks_t, fn):
    """Point the McpPolicy at the policy tensors and check the batch; returns (states, masks, tensors to keep alive)."""
    x = _c(x, "states")
    if x.dim() != 2 or x.shape[1] != pst.Ds:
        raise RuntimeError("%s: states must be [M, %d]" % (fn, pst.Ds))
    M = x.shape[0]
    keep = [_c(tens[k], k) for k in ("log_ls", "centers", "W")]
    pst.log_ls, pst.centers, pst.W = (k.data_ptr() for k in keep)
    b = _c(tens["bias"], "bias") if tens.get("bias") is not None else None
    tr = _c(tens["target_traj"], "target_traj") if tens.get("target_traj") is not None else None
    if tr is not None and not (0 <= int(t) < tr.shape[0]):
        raise RuntimeError("%s: time index %s outside the target trajectory" % (fn, t))
    pst.bias = b.data_ptr() if b is not None else None
    pst.target_traj = tr.data_ptr() if tr is not None else None
    mk = None
    if masks_t is not None:
        mk = masks_t.detach().to(torch.uint8).contiguous()
        if not mk.is_cuda or tuple(mk.shape) != (M, pst.nb):
            raise RuntimeError("%s: masks must be a CUDA tensor [M, nb]" % fn)
    return x, mk, keep + [b, tr]


@_restores_device
def policy_forward(pst, tens, x, t=0, p_dropout=0.0, masks_t=None, seed=0, particle_offset=0):
    """u = pi(x) for a batch of states through the CUDA policy kernel.  Policy.py:242-265,323-335,389-403."""
    x, mk, _keep = _policy_call_args(pst, tens, x, t, masks_t, "policy_forward")
    L = _enter(x.device)
    M = x.shape[0]
    u = torch.empty(M, pst.Du, dtype=F64, device=x.device)
    N.check(L.mcpilco_policy_forward(C.byref(pst), M, int(t or 0), _ptr(x), float(p_dropout), _ptr(mk), int(seed), int(particle_offset),
                                     _ptr(u), _stream(x.device)))
    return u


@_restores_device
def policy_backward(pst, tens, x, g_u, t=0, p_dropout=0.0, masks_t=None, seed=0, particle_offset=0, want_gx=True):
    """Vector-Jacobian product of policy_forward with the same arguments: {"log_ls" [1, Dp], "centers" [nb, Dp], "W" [Du, nb],
    "bias" [Du] or None, "x" [M, Ds] or None} = g_u^T d pi(x) / d(.).  The dropout mask is the forward's (the same masks_t, or the
    same Philox draws for the same seed and particle_offset)."""
    x, mk, _keep = _policy_call_args(pst, tens, x, t, masks_t, "policy_backward")
    L = _enter(x.device)
    M, dev = x.shape[0], x.device
    g_u = _c(g_u, "grad_u")
    if tuple(g_u.shape) != (M, pst.Du):
        raise RuntimeError("policy_backward: grad_u must be [%d, %d]" % (M, pst.Du))
    out = {"log_ls": torch.empty(1, pst.Dp, dtype=F64, device=dev), "centers": torch.empty(pst.nb, pst.Dp, dtype=F64, device=dev),
           "W": torch.empty(pst.Du, pst.nb, dtype=F64, device=dev),
           "bias": torch.empty(pst.Du, dtype=F64, device=dev) if pst.has_bias else None,
           "x": torch.empty(M, pst.Ds, dtype=F64, device=dev) if want_gx else None}
    wsb = L.mcpilco_policy_backward_workspace_bytes(M, pst.nb, pst.Dp, pst.Du)
    ws = _workspace(dev, wsb, "policy_bwd")
    N.check(L.mcpilco_policy_backward(C.byref(pst), M, int(t or 0), _ptr(x), float(p_dropout), _ptr(mk), int(seed), int(particle_offset),
                                      _ptr(g_u), _ptr(out["x"]), _ptr(out["log_ls"]), _ptr(out["centers"]), _ptr(out["W"]), _ptr(out["bias"]),
                                      _ptr(ws), ws.numel(), _stream(dev)))
    return out


@_restores_device
def init_particles(kind, a, b, M, seed=0, particle_offset=0, seed_dev=None):
    """Initial particles keyed by the global particle id.  kind "gauss": a = mean(s) [n_modes, Ds], b = std(s);
    kind "uniform": a = lower, b = upper bound.  MC_PILCO.py:635-657."""
    a, b = _c(a, "a").reshape(-1, a.shape[-1]), _c(b, "b").reshape(-1, b.shape[-1])
    L = _enter(a.device)
    x0 = torch.empty(int(M), a.shape[1], dtype=F64, device=a.device)
    N.check(L.mcpilco_init_particles(0 if kind == "gauss" else 1, _ptr(a), _ptr(b), a.shape[0], int(M), a.shape[1], int(seed),
                                     int(particle_offset), _ptr(seed_dev), _ptr(x0), _stream(a.device)))
    return x0


def prof_enable(on=True):
    N.check(N.lib().mcpilco_prof_enable(1 if on else 0))


def prof_read():
    ms, n, fl = C.c_double(0), C.c_uint64(0), C.c_double(0)
    N.check(N.lib().mcpilco_prof_read(C.byref(ms), C.byref(n), C.byref(fl)))
    return ms.value, int(n.value), fl.value


@_restores_device
def ozaki_matmul(A, B, slices=8):
    """A [M, N] @ B[N, N]^T through the INT8 tensor-core contraction (test / benchmark hook)."""
    A, B = _c(A, "A"), _c(B, "B")
    L = _enter(A.device)
    M, Nn = A.shape
    planes = torch.empty(L.mcpilco_ozaki_plane_bytes(Nn, slices), dtype=torch.uint8, device=A.device)
    pexp = torch.empty(Nn, dtype=torch.int32, device=A.device)
    N.check(L.mcpilco_ozaki_prepare(_ptr(B), Nn, B.stride(0), slices, _ptr(planes), _ptr(pexp), _stream(A.device)))
    V = torch.empty(M, Nn, dtype=F64, device=A.device)
    sb = L.mcpilco_ozaki_scratch_bytes(M, Nn, slices)
    scratch = torch.empty(sb, dtype=torch.uint8, device=A.device)
    N.check(L.mcpilco_ozaki_contract(_ptr(A), A.stride(0), M, Nn, slices, _ptr(planes), _ptr(pexp), _ptr(V), Nn, _ptr(scratch), sb,
                                     _stream(A.device)))
    return V, planes, pexp
