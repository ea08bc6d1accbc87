"""`torch.ops.mcpilco.*` — the GP operators of the hot path registered as torch custom ops (torch.library), a thin layer over the C ABI.

Custom ops take tensors and scalars only, so a kernel specification travels as a CPU uint8 tensor holding the bytes of the POD
`McpGpSpec` (`spec_tensor(spec)` / `GP_prior.gp_spec(D)`).  CUDA float64 tensors only; there is no CPU implementation to dispatch to.

    torch.ops.mcpilco.gp_covariance(spec, X1, X2, add_noise) -> K
    torch.ops.mcpilco.gp_diag_covariance(spec, X) -> diag
    torch.ops.mcpilco.gp_precompute(spec, X, y) -> (alpha [N,1], Kinv [N,N])
    torch.ops.mcpilco.gp_predict(spec, Xtr, alpha, Kinv, Xs, var_scale) -> (mean [M,1], var [M,1])
    torch.ops.mcpilco.gp_predict_jac(spec, Xtr, alpha, Kinv, Xs, var_scale) -> (mean, var, dmean/dx [M,D], dvar/dx [M,D])
    torch.ops.mcpilco.gp_nlml(spec, X, y) -> packed value + gradient (layout: include/mcpilco_b200.h)

    torch.ops.mcpilco.policy_forward(pol, log_ls, centers, W, bias, target_traj, x, t, p_dropout, masks_t, seed, particle_offset) -> u
    torch.ops.mcpilco.policy_backward(<the same arguments>, grad_u, want_gx) -> (g_log_ls, g_centers, g_W, g_bias, g_x)

gp_predict and policy_forward are differentiable once (register_autograd): gp_predict w.r.t. Xs only (the fitted GP receives no
gradient), policy_forward w.r.t. log_ls, centers, W, bias and x through policy_backward, which redraws the forward's dropout mask from
the saved seed (or takes the same masks_t).  A policy travels as a CPU uint8 tensor with the bytes of McpPolicy (`policy_tensor`).

    torch.ops.mcpilco.rollout_fwd(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0,
                                  eps, masks, meas_eps, seed_dev, need_grad) -> (states, inputs, cost[2], cost_stats[H,2], jac, pol_in)
    torch.ops.mcpilco.rollout_bwd(<the same leading arguments>, states, inputs, jac, pol_in, grad_cost, grad_states, grad_inputs,
                                  want_gx0) -> (g_log_ls, g_centers, g_W, g_bias, g_x0)

The rollout's POD descriptors (McpModel, McpPolicy, McpCost, McpMeas, the scalars of McpRollout / McpNoise) travel as ONE CPU uint8
tensor (`rollout_descriptor`), the E fitted GPs as a CPU uint8 tensor of their McpGpSpec bytes, a CPU float64 tensor of per-GP scalars
and a flat list of device tensors (`gp_pack`).  `RolloutCall` bundles those arguments; the autograd node of the class API
(policy_learning.MC_PILCO._ParticleRollout) and the captured optimisation step run on these two ops.
"""
import ctypes as C
import struct
from typing import List, Optional, Tuple

import torch

from . import _native as N
from . import _ops as ops


def spec_tensor(spec):
    """CPU uint8 tensor with the bytes of a McpGpSpec."""
    return torch.frombuffer(bytearray(C.string_at(C.addressof(spec), C.sizeof(spec))), dtype=torch.uint8).clone()


def _spec(t):
    if t.device.type != "cpu" or t.dtype != torch.uint8 or t.numel() != C.sizeof(N.GpSpec):
        raise RuntimeError("mcpilco: spec must be a CPU uint8 tensor of %d bytes (torch_ops.spec_tensor)" % C.sizeof(N.GpSpec))
    return N.GpSpec.from_buffer_copy(bytes(t.contiguous().numpy().tobytes()))


@torch.library.custom_op("mcpilco::gp_covariance", mutates_args=(), device_types="cuda")
def gp_covariance(spec: torch.Tensor, X1: torch.Tensor, X2: Optional[torch.Tensor], add_noise: bool) -> torch.Tensor:
    return ops.gp_covariance(_spec(spec), X1, X2, add_noise)


@torch.library.custom_op("mcpilco::gp_diag_covariance", mutates_args=(), device_types="cuda")
def gp_diag_covariance(spec: torch.Tensor, X: torch.Tensor) -> torch.Tensor:
    return ops.gp_diag_covariance(_spec(spec), X)


@torch.library.custom_op("mcpilco::gp_precompute", mutates_args=(), device_types="cuda")
def gp_precompute(spec: torch.Tensor, X: torch.Tensor, y: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    alpha, Kinv = ops.gp_precompute(_spec(spec), X, y)
    return alpha, Kinv.contiguous()


@torch.library.custom_op("mcpilco::gp_predict", mutates_args=(), device_types="cuda")
def gp_predict(spec: torch.Tensor, Xtr: torch.Tensor, alpha: torch.Tensor, Kinv: torch.Tensor, Xs: torch.Tensor,
               var_scale: float) -> Tuple[torch.Tensor, torch.Tensor]:
    mean, var = ops._gp_predict([ops.FittedGp(_spec(spec), Xtr, alpha, Kinv, var_scale=var_scale)], Xs)
    return mean, var


@torch.library.custom_op("mcpilco::gp_predict_jac", mutates_args=(), device_types="cuda")
def gp_predict_jac(spec: torch.Tensor, Xtr: torch.Tensor, alpha: torch.Tensor, Kinv: torch.Tensor, Xs: torch.Tensor,
                   var_scale: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    mean, var, jm, jv = ops._gp_predict([ops.FittedGp(_spec(spec), Xtr, alpha, Kinv, var_scale=var_scale)], Xs, jac=True)
    return mean, var, jm[:, 0, :].contiguous(), jv[:, 0, :].contiguous()


@torch.library.custom_op("mcpilco::gp_nlml", mutates_args=(), device_types="cuda")
def gp_nlml(spec: torch.Tensor, X: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    return ops.gp_nlml(_spec(spec), X, y)


# shape functions so the ops compose with tracing / fake tensors
@gp_covariance.register_fake
def _(spec, X1, X2, add_noise):
    return X1.new_empty(X1.shape[0], X1.shape[0] if X2 is None else X2.shape[0])


@gp_diag_covariance.register_fake
def _(spec, X):
    return X.new_empty(X.shape[0])


@gp_precompute.register_fake
def _(spec, X, y):
    return X.new_empty(X.shape[0], 1), X.new_empty(X.shape[0], X.shape[0])


@gp_predict.register_fake
def _(spec, Xtr, alpha, Kinv, Xs, var_scale):
    return Xs.new_empty(Xs.shape[0], 1), Xs.new_empty(Xs.shape[0], 1)


@gp_predict_jac.register_fake
def _(spec, Xtr, alpha, Kinv, Xs, var_scale):
    return Xs.new_empty(Xs.shape[0], 1), Xs.new_empty(Xs.shape[0], 1), Xs.new_empty(Xs.shape), Xs.new_empty(Xs.shape)


@gp_nlml.register_fake
def _(spec, X, y):
    return X.new_empty(4 + N.MAX_D + N.MAX_POLY * N.MAX_DEG * (N.MAX_D + 1))


def _no_double_backward(name):
    if torch.is_grad_enabled():
        raise RuntimeError("mcpilco: %s is differentiable once; double backward (create_graph=True) is not supported" % name)


# d/dXs of the posterior (the fitted GP itself receives no gradient): the backward recomputes the Jacobians through gp_predict_jac
def _gp_predict_setup(ctx, inputs, output):
    ctx.args = inputs


def _gp_predict_backward(ctx, g_mean, g_var):
    _no_double_backward("mcpilco::gp_predict")
    spec, Xtr, alpha, Kinv, Xs, var_scale = ctx.args
    if not ctx.needs_input_grad[4]:
        return None, None, None, None, None, None
    _, _, jm, jv = gp_predict_jac(spec, Xtr, alpha, Kinv, Xs, var_scale)
    return None, None, None, None, ops.gp_predict_vjp(jm.unsqueeze(1), jv.unsqueeze(1), g_mean, g_var), None


gp_predict.register_autograd(_gp_predict_backward, setup_context=_gp_predict_setup)


# ---------------------------------------------------------------------------------------------------------------------
# the stand-alone policy (Sum_of_gaussians.forward, Policy.py:242-265,323-335,389-403) and its vector-Jacobian product
# ---------------------------------------------------------------------------------------------------------------------
def policy_tensor(pst):
    """CPU uint8 tensor with the bytes of a McpPolicy (its pointer fields are re-pointed at the tensor arguments on every call)."""
    return torch.frombuffer(bytearray(_bytes_of(pst)), dtype=torch.uint8).clone()


def _policy(t):
    if t.device.type != "cpu" or t.dtype != torch.uint8 or t.numel() != C.sizeof(N.Policy):
        raise RuntimeError("mcpilco: policy must be a CPU uint8 tensor of %d bytes (torch_ops.policy_tensor)" % C.sizeof(N.Policy))
    return N.Policy.from_buffer_copy(bytes(t.contiguous().numpy().tobytes()))


def _ptens(log_ls, centers, W, bias, target_traj):
    return {"log_ls": log_ls, "centers": centers, "W": W, "bias": bias, "target_traj": target_traj}


@torch.library.custom_op("mcpilco::policy_forward", mutates_args=(), device_types="cuda")
def policy_forward(pol: torch.Tensor, log_ls: torch.Tensor, centers: torch.Tensor, W: torch.Tensor, bias: Optional[torch.Tensor],
                   target_traj: Optional[torch.Tensor], x: torch.Tensor, t: int, p_dropout: float, masks_t: Optional[torch.Tensor],
                   seed: int, particle_offset: int) -> torch.Tensor:
    return ops.policy_forward(_policy(pol), _ptens(log_ls, centers, W, bias, target_traj), x, t=t, p_dropout=p_dropout, masks_t=masks_t,
                              seed=seed, particle_offset=particle_offset)


@torch.library.custom_op("mcpilco::policy_backward", mutates_args=(), device_types="cuda")
def policy_backward(pol: torch.Tensor, log_ls: torch.Tensor, centers: torch.Tensor, W: torch.Tensor, bias: Optional[torch.Tensor],
                    target_traj: Optional[torch.Tensor], x: torch.Tensor, t: int, p_dropout: float, masks_t: Optional[torch.Tensor],
                    seed: int, particle_offset: int, grad_u: torch.Tensor,
                    want_gx: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    g = ops.policy_backward(_policy(pol), _ptens(log_ls, centers, W, bias, target_traj), x, grad_u, t=t, p_dropout=p_dropout, masks_t=masks_t,
                            seed=seed, particle_offset=particle_offset, want_gx=want_gx)
    none = lambda: x.new_empty(0)  # noqa: E731
    return g["log_ls"], g["centers"], g["W"], g["bias"] if g["bias"] is not None else none(), g["x"] if g["x"] is not None else none()


@policy_forward.register_fake
def _(pol, log_ls, centers, W, bias, target_traj, x, t, p_dropout, masks_t, seed, particle_offset):
    return x.new_empty(x.shape[0], W.shape[0])


@policy_backward.register_fake
def _(pol, log_ls, centers, W, bias, target_traj, x, t, p_dropout, masks_t, seed, particle_offset, grad_u, want_gx):
    e = x.new_empty
    return e(log_ls.shape), e(centers.shape), e(W.shape), e(W.shape[0] if bias is not None else 0), e(x.shape if want_gx else 0)


def _policy_setup(ctx, inputs, output):
    ctx.args = inputs  # the seed among them: the backward redraws the forward's Philox dropout mask


def _policy_backward(ctx, grad_u):
    _no_double_backward("mcpilco::policy_forward")
    pol, log_ls, centers, W, bias, target_traj, x, t, p_dropout, masks_t, seed, particle_offset = ctx.args
    need = ctx.needs_input_grad
    gl, gc, gw, gb, gx = policy_backward(pol, log_ls.detach(), centers.detach(), W.detach(), None if bias is None else bias.detach(),
                                         target_traj, x.detach(), t, p_dropout, masks_t, seed, particle_offset, grad_u.contiguous(),
                                         bool(need[6]))
    return (None, gl.reshape(log_ls.shape) if need[1] else None, gc if need[2] else None, gw if need[3] else None,
            gb if (bias is not None and need[4]) else None, None, gx.reshape(x.shape) if need[6] else None, None, None, None, None, None)


policy_forward.register_autograd(_policy_backward, setup_context=_policy_setup)


# ---------------------------------------------------------------------------------------------------------------------
# the particle rollout as two ops (SURVEY.md 8b): MC_PILCO.apply_policy (MC_PILCO.py:615-674, :808-906) and the autograd pass of
# cost.backward() (MC_PILCO.py:522)
# ---------------------------------------------------------------------------------------------------------------------
_DESC_TAIL = "<iiiidQQ"  # M, H, M_global, pad, p_dropout, seed, particle_offset


def _bytes_of(st):
    return C.string_at(C.addressof(st), C.sizeof(st))


def rollout_descriptor(model, policy, cost, meas, M, H, p_dropout, seed, particle_offset, M_global):
    """CPU uint8 tensor: McpModel | McpPolicy | McpCost | McpMeas (pointer fields ignored) | M, H, M_global, p_dropout, seed, offset."""
    cost = cost if cost is not None else N.Cost()
    meas = meas if meas is not None else N.Meas()
    raw = _bytes_of(model) + _bytes_of(policy) + _bytes_of(cost) + _bytes_of(meas) + struct.pack(
        _DESC_TAIL, int(M), int(H), int(M_global), 0, float(p_dropout), int(seed) & ((1 << 64) - 1), int(particle_offset))
    return torch.frombuffer(bytearray(raw), dtype=torch.uint8).clone()


def _parse_descriptor(desc):
    if desc.device.type != "cpu" or desc.dtype != torch.uint8:
        raise RuntimeError("mcpilco: the rollout descriptor must be a CPU uint8 tensor (torch_ops.rollout_descriptor)")
    raw = bytes(desc.contiguous().numpy().tobytes())
    sizes = [C.sizeof(N.Model), C.sizeof(N.Policy), C.sizeof(N.Cost), C.sizeof(N.Meas), struct.calcsize(_DESC_TAIL)]
    if len(raw) != sum(sizes):
        raise RuntimeError("mcpilco: rollout descriptor has %d bytes, expected %d" % (len(raw), sum(sizes)))
    off, parts = 0, []
    for cls, n in zip((N.Model, N.Policy, N.Cost, N.Meas), sizes):
        parts.append(cls.from_buffer_copy(raw[off:off + n]))
        off += n
    M, H, Mg, _, p_drop, seed, offset = struct.unpack(_DESC_TAIL, raw[off:])
    return parts + [M, H, Mg, p_drop, seed, offset]


def gp_pack(gps):
    """(specs uint8 CPU [E, sizeof(McpGpSpec)], scalars float64 CPU [E, 6], tensors) for a list of ops.FittedGp.  Six device tensors per
    GP: Xtr, alpha, Kinv, Linv, digit planes, plane exponents (absent ones are empty tensors)."""
    dev = gps[0].Xtr.device
    e64, e8, e32 = (torch.empty(0, dtype=d, device=dev) for d in (torch.float64, torch.uint8, torch.int32))
    specs = torch.stack([spec_tensor(g.spec) for g in gps])
    scal = torch.tensor([[g.var_scale, float(g.ozaki), g.kdiag_max, float(g.ld), float(g.ld_linv), 0.0] for g in gps], dtype=torch.float64)
    tens = []
    for g in gps:
        tens += [g.Xtr, g.alpha, g.Kinv, g.Linv if g.Linv is not None else e64, g.planes if g.planes is not None else e8,
                 g.plane_exp if g.plane_exp is not None else e32]
    return specs, scal, tens


def _unpack_gps(specs, scal, tens):
    gps = []
    for e in range(specs.shape[0]):
        X, a, K, Li, pl, pe = tens[6 * e:6 * e + 6]
        vs, oz, kd, ld, ldl, _ = (float(v) for v in scal[e])
        gps.append(ops.FittedGp.from_parts(_spec(specs[e]), X, a, K, int(ld), vs, int(oz), pl if pl.numel() else None,
                                           pe if pe.numel() else None, Li if Li.numel() else None, int(ldl), kd))
    return gps


def _plan(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0, eps, masks, meas_eps, seed_dev,
          need_grad, buffers=None):
    model, policy, cost, meas, M, H, Mg, p_drop, seed, offset = _parse_descriptor(desc)
    pt = {"log_ls": log_ls, "centers": centers, "W": W, "bias": bias, "target_traj": policy_traj}
    return ops.RolloutPlan(model, _unpack_gps(gp_specs, gp_scalars, gp_tensors), policy, pt, cost=cost, cost_traj=cost_traj, meas=meas, M=M,
                           H=H, p_dropout=p_drop, seed=seed, particle_offset=offset, need_grad=need_grad, eps=eps, masks=masks,
                           meas_eps=meas_eps, device=x0.device, M_global=Mg, seed_dev=seed_dev, buffers=buffers)


@torch.library.custom_op("mcpilco::rollout_fwd", mutates_args=(), device_types="cuda")
def rollout_fwd(desc: torch.Tensor, gp_specs: torch.Tensor, gp_scalars: torch.Tensor, gp_tensors: List[torch.Tensor], log_ls: torch.Tensor,
                centers: torch.Tensor, W: torch.Tensor, bias: Optional[torch.Tensor], policy_traj: Optional[torch.Tensor],
                cost_traj: Optional[torch.Tensor], x0: torch.Tensor, eps: Optional[torch.Tensor], masks: Optional[torch.Tensor],
                meas_eps: Optional[torch.Tensor], seed_dev: Optional[torch.Tensor],
                need_grad: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    plan = _plan(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0, eps, masks, meas_eps, seed_dev,
                 need_grad)
    states, inputs = plan.forward(x0)
    none = lambda: x0.new_empty(0)  # noqa: E731  (a fresh tensor per absent output: returns of a custom op must not alias each other)
    return (states, inputs, plan.cost_out if plan.cost_out is not None else none(), plan.cost_stats if plan.cost_stats is not None else none(),
            plan.jac if plan.jac is not None else none(), plan.pol_in if plan.pol_in is not None else none())


@torch.library.custom_op("mcpilco::rollout_bwd", mutates_args=(), device_types="cuda")
def rollout_bwd(desc: torch.Tensor, gp_specs: torch.Tensor, gp_scalars: torch.Tensor, gp_tensors: List[torch.Tensor], log_ls: torch.Tensor,
                centers: torch.Tensor, W: torch.Tensor, bias: Optional[torch.Tensor], policy_traj: Optional[torch.Tensor],
                cost_traj: Optional[torch.Tensor], x0: torch.Tensor, eps: Optional[torch.Tensor], masks: Optional[torch.Tensor],
                meas_eps: Optional[torch.Tensor], seed_dev: Optional[torch.Tensor], states: torch.Tensor, inputs: torch.Tensor,
                jac: torch.Tensor, pol_in: torch.Tensor, grad_cost: float, grad_states: Optional[torch.Tensor],
                grad_inputs: Optional[torch.Tensor],
                want_gx0: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    bufs = {"states": states, "inputs": inputs, "jac": jac if jac.numel() else None, "pol_in": pol_in if pol_in.numel() else None}
    plan = _plan(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0, eps, masks, meas_eps, seed_dev,
                 True, buffers=bufs)
    plan.x0 = x0
    plan.r.x0 = x0.data_ptr()
    g = plan.backward(grad_cost=grad_cost, grad_states=grad_states, grad_inputs=grad_inputs, want_gx0=want_gx0)
    none = lambda: x0.new_empty(0)  # noqa: E731
    return g["log_ls"], g["centers"], g["W"], g["bias"] if g["bias"] is not None else none(), g["x0"] if g["x0"] is not None else none()


@rollout_fwd.register_fake
def _(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0, eps, masks, meas_eps, seed_dev, need_grad):
    model, policy, cost, meas, M, H, Mg, p_drop, seed, offset = _parse_descriptor(desc)
    e = x0.new_empty
    return (e(H, M, model.Ds), e(H, M, model.Du), e(2 if cost.kind else 0), e((H, 2) if cost.kind else 0),
            e((max(H - 1, 1), M, model.E, model.D) if need_grad else 0), e((H, M, model.Ds) if meas.enabled else 0))


@rollout_bwd.register_fake
def _(desc, gp_specs, gp_scalars, gp_tensors, log_ls, centers, W, bias, policy_traj, cost_traj, x0, eps, masks, meas_eps, seed_dev, states,
      inputs, jac, pol_in, grad_cost, grad_states, grad_inputs, want_gx0):
    e = x0.new_empty
    return e(log_ls.shape), e(centers.shape), e(W.shape), e(W.shape[0] if bias is not None else 0), e(x0.shape if want_gx0 else 0)


class RolloutCall:
    """The argument bundle of one rollout for the two ops above, built once per apply_policy from the class-level objects."""

    def __init__(self, model, gps, policy, pol_tensors, cost=None, cost_traj=None, meas=None, M=1, H=1, p_dropout=0.0, seed=0,
                 particle_offset=0, eps=None, masks=None, meas_eps=None, M_global=0, seed_dev=None):
        self.M, self.H, self.has_cost = int(M), int(H), cost is not None and cost.kind != 0
        self.desc = rollout_descriptor(model, policy, cost, meas, M, H, p_dropout, seed, particle_offset, M_global)
        self.gp_specs, self.gp_scalars, self.gp_tensors = gp_pack(gps)
        as8 = lambda m: None if m is None else m.detach().to(torch.uint8).contiguous()  # noqa: E731
        c = lambda t: None if t is None else t.detach().contiguous()  # noqa: E731
        self.head = (pol_tensors["log_ls"], pol_tensors["centers"], pol_tensors["W"], pol_tensors.get("bias"), c(pol_tensors.get("target_traj")),
                     c(cost_traj))
        self.noise = (c(eps), as8(masks), c(meas_eps), seed_dev)

    def _args(self, x0):
        det = lambda t: None if t is None else t.detach()  # noqa: E731
        return (self.desc, self.gp_specs, self.gp_scalars, self.gp_tensors) + tuple(det(t) for t in self.head) + (x0.detach().contiguous(),) + self.noise

    def forward(self, x0, need_grad):
        """-> states, inputs, cost_out [2] or None, cost_stats [H, 2] or None, jac, pol_in (empty tensors when absent)"""
        st, inp, cost, stats, jac, pol_in = torch.ops.mcpilco.rollout_fwd(*self._args(x0), bool(need_grad))
        return st, inp, (cost if cost.numel() else None), (stats if stats.numel() else None), jac, pol_in

    def backward(self, x0, states, inputs, jac, pol_in, grad_cost=0.0, grad_states=None, grad_inputs=None, want_gx0=False):
        c = lambda t: None if t is None else t.detach().contiguous()  # noqa: E731
        g = torch.ops.mcpilco.rollout_bwd(*self._args(x0), states, inputs, jac, pol_in, float(grad_cost), c(grad_states), c(grad_inputs),
                                          bool(want_gx0))
        return {"log_ls": g[0], "centers": g[1], "W": g[2], "bias": g[3] if g[3].numel() else None, "x0": g[4] if g[4].numel() else None}
