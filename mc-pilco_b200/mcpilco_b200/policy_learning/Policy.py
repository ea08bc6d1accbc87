"""Control policies — the reference's `policy_learning/Policy.py` surface for the rollout hot path: Policy (:14-72),
Sum_of_gaussians (:153-265), Sum_of_gaussians_with_angles (:268-335), Sum_of_gaussians_with_target_trajectory (:338-403).

  z = feat(x) / scale_factor ;  d_b = sum_j ((z_j - c_bj) / l_j)^2 ;  h = dropout(exp(-d), p)  (kept units scaled by 1/(1-p)) ;
  u = u_max * tanh((W h + bias) / u_max)

Parameter names (`log_lengthscales`, `centers`, `f_linear.weight`, `f_linear.bias`) are the reference's, so state_dicts load
unchanged and `cost.backward()` fills the same `.grad` fields.  Inside a particle rollout the policy is evaluated by the fused
CUDA kernels (MC_PILCO.apply_policy); calling the module on a batch of states runs the same CUDA policy kernel stand-alone.
A stand-alone call is differentiable (once) w.r.t. the parameters and the states: its backward is the CUDA vector-Jacobian product
`torch.ops.mcpilco.policy_backward`, with the forward's dropout mask.  Under `torch.no_grad()`, or when nothing involved requires
grad, no graph is recorded.  Exploration policies and PD_controller act on the real system one state at a time
and are outside the hot path (SURVEY.md §2 row 7).
"""
import numpy as np
import torch

from .. import _ops as ops
from .. import _pack as P
from .. import torch_ops as TO


class Policy(torch.nn.Module):
    """Superclass of the policies (reference :14-72)."""

    def __init__(self, state_dim, input_dim, flg_squash=False, u_max=1, dtype=torch.float64, device=torch.device("cpu")):
        super().__init__()
        self.state_dim, self.input_dim = state_dim, input_dim
        self.dtype, self.device = dtype, device
        self.flg_squash, self.u_max = flg_squash, u_max
        self.f_squash = (lambda x: self.squashing(x, u_max)) if flg_squash else (lambda x: x)

    def forward(self, states, t=None, p_dropout=0.0):
        raise NotImplementedError()

    def forward_np(self, state, t=None):
        out = self(states=torch.tensor(state, dtype=self.dtype, device=self.device), t=t)
        return out.detach().cpu().numpy()

    def to(self, device):
        super().to(device)
        self.device = device

    def squashing(self, u, u_max):
        """u_max * tanh(u / u_max), element-wise bound per input (reference :52-60)."""
        if not np.isscalar(u_max):
            u_max = torch.tensor(u_max, dtype=self.dtype, device=u.device)
        return u_max * torch.tanh(u / u_max)

    def get_np_policy(self):
        return lambda state, t: self.forward_np(state, t)

    def reinit(self, scaling=1):
        raise NotImplementedError()


class Sum_of_gaussians(Policy):
    """RBF-network policy with dropout and tanh squashing (reference :153-265)."""

    _kind = "plain"

    def __init__(self, state_dim, input_dim, num_basis, flg_train_lengthscales=True, lengthscales_init=None, flg_train_centers=True,
                 centers_init=None, centers_init_min=-1, centers_init_max=1, weight_init=None, flg_train_weight=True, flg_bias=False,
                 bias_init=None, flg_train_bias=False, flg_squash=False, u_max=1, scale_factor=None, flg_drop=True,
                 dtype=torch.float64, device=torch.device("cpu")):
        super().__init__(state_dim=state_dim, input_dim=input_dim, flg_squash=flg_squash, u_max=u_max, dtype=dtype, device=device)
        self.num_basis = num_basis
        if lengthscales_init is None:
            lengthscales_init = np.ones(state_dim)
        self.log_lengthscales = torch.nn.Parameter(torch.tensor(np.log(lengthscales_init), dtype=dtype, device=device).reshape([1, -1]),
                                                   requires_grad=flg_train_lengthscales)
        if centers_init is None:
            centers_init = centers_init_min + (centers_init_max - centers_init_min) * np.random.rand(num_basis, state_dim)
        self.centers = torch.nn.Parameter(torch.tensor(centers_init, dtype=dtype, device=device), requires_grad=flg_train_centers)
        self.f_linear = torch.nn.Linear(in_features=num_basis, out_features=input_dim, bias=flg_bias)
        w = np.ones([input_dim, num_basis]) if weight_init is None else weight_init
        self.f_linear.weight.data = torch.tensor(np.asarray(w), dtype=dtype, device=device).reshape(input_dim, num_basis)
        self.f_linear.weight.requires_grad = flg_train_weight
        if flg_bias:
            self.f_linear.bias.requires_grad = flg_train_bias
            if bias_init is not None:
                self.f_linear.bias.data = torch.tensor(np.asarray(bias_init), dtype=dtype, device=device).reshape(input_dim)
        self.f_linear.type(dtype)
        self.f_linear.to(device)
        self.flg_bias = flg_bias
        if scale_factor is None:
            scale_factor = np.ones(state_dim)
        self.scale_factor = torch.tensor(scale_factor, dtype=dtype, device=device).reshape([1, -1])
        self.flg_drop = bool(flg_drop)
        # kept for API compatibility with code that swaps the dropout function (the fused kernels use flg_drop)
        self.f_drop = torch.nn.functional.dropout if flg_drop else (lambda x, p: x)

    def reinit(self, lenghtscales_par, centers_par, weight_par):
        """Re-draw centres / weights uniformly around zero (reference :229-240); `lenghtscales_par` [sic]."""
        dev = self.centers.device
        self.log_lengthscales.data = torch.tensor(np.log(lenghtscales_par), dtype=self.dtype, device=dev).reshape([1, -1])
        self.centers.data = (torch.tensor(centers_par, dtype=self.dtype, device=dev) * 2
                             * (torch.rand(self.num_basis, self.state_dim, dtype=self.dtype, device=dev) - 0.5))
        self.f_linear.weight.data = weight_par * (torch.rand(self.input_dim, self.num_basis, dtype=self.dtype, device=dev) - 0.5)

    # ---- what the fused rollout consumes ------------------------------------------------------------------------
    def _raw_state_dim(self):
        return self.state_dim

    def policy_struct(self):
        return P.policy_struct(self._kind, self.num_basis, self.state_dim, self.input_dim, self._raw_state_dim(),
                               u_max=self.u_max if self.flg_squash else None, scale=self.scale_factor,
                               angle=getattr(self, "angle_indices", ()), non_angle=getattr(self, "non_angle_indices", ()),
                               has_bias=self.flg_bias, use_drop=self.flg_drop)

    def policy_tensors(self):
        return {"log_ls": self.log_lengthscales, "centers": self.centers, "W": self.f_linear.weight,
                "bias": self.f_linear.bias if self.flg_bias else None, "target_traj": getattr(self, "target_traj", None)}

    def forward(self, states, t=None, p_dropout=0.0):
        """u = pi(states) through the CUDA policy kernel; dropout masks come from a Philox stream seeded from torch's RNG.  With grad
        mode on and the states or a parameter requiring grad, the call is recorded for autograd (once differentiable)."""
        x = states.reshape([-1, self._raw_state_dim()])
        seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if (self.flg_drop and p_dropout > 0.0) else 0
        tens = self.policy_tensors()
        t = 0 if t is None else t
        if torch.is_grad_enabled() and any(v is not None and v.requires_grad for v in (x, tens["log_ls"], tens["centers"], tens["W"], tens["bias"])):
            traj = tens["target_traj"]
            return torch.ops.mcpilco.policy_forward(TO.policy_tensor(self.policy_struct()), tens["log_ls"], tens["centers"], tens["W"],
                                                    tens["bias"], None if traj is None else traj.detach(), x, int(t), float(p_dropout), None,
                                                    seed, 0)
        return ops.policy_forward(self.policy_struct(), tens, x, t=t, p_dropout=p_dropout, seed=seed)


class Sum_of_gaussians_with_angles(Sum_of_gaussians):
    """Policy input [x[non_angle], cos x[angle], sin x[angle]] — cos BEFORE sin (reference :268-335)."""

    _kind = "angles"

    def __init__(self, state_dim, input_dim, num_basis, angle_indices, non_angle_indices, flg_train_lengthscales=True,
                 lengthscales_init=None, flg_train_centers=True, centers_init=None, centers_init_min=-1, centers_init_max=1,
                 weight_init=None, flg_train_weight=True, flg_bias=False, bias_init=None, flg_train_bias=False, flg_squash=False, u_max=1,
                 flg_drop=True, dtype=torch.float64, device=torch.device("cpu")):
        self.angle_indices = np.asarray(angle_indices)
        self.non_angle_indices = np.asarray(non_angle_indices)
        self.num_angle_indices = self.angle_indices.size
        self.num_non_angle_indices = self.non_angle_indices.size
        super().__init__(state_dim=state_dim + self.num_angle_indices, input_dim=input_dim, num_basis=num_basis,
                         flg_train_lengthscales=flg_train_lengthscales, lengthscales_init=lengthscales_init,
                         flg_train_centers=flg_train_centers, centers_init=centers_init, centers_init_min=centers_init_min,
                         centers_init_max=centers_init_max, weight_init=weight_init, flg_train_weight=flg_train_weight, flg_bias=flg_bias,
                         bias_init=bias_init, flg_train_bias=flg_train_bias, flg_squash=flg_squash, u_max=u_max, flg_drop=flg_drop,
                         dtype=dtype, device=device)

    def _raw_state_dim(self):
        return self.state_dim - self.num_angle_indices


class Sum_of_gaussians_with_target_trajectory(Sum_of_gaussians):
    """Policy input [x, target_t - x]; `state_dim` is the EXTENDED dimension 2*Ds (reference :338-403)."""

    _kind = "target"

    def __init__(self, state_dim, input_dim, num_basis, target_traj, flg_train_lengthscales=True, lengthscales_init=None,
                 flg_train_centers=True, centers_init=None, centers_init_min=-1, centers_init_max=1, weight_init=None,
                 flg_train_weight=True, flg_bias=False, bias_init=None, flg_train_bias=False, flg_squash=False, u_max=1, flg_drop=True,
                 dtype=torch.float64, device=torch.device("cpu")):
        super().__init__(state_dim=state_dim, input_dim=input_dim, num_basis=num_basis, flg_train_lengthscales=flg_train_lengthscales,
                         lengthscales_init=lengthscales_init, flg_train_centers=flg_train_centers, centers_init=centers_init,
                         centers_init_min=centers_init_min, centers_init_max=centers_init_max, weight_init=weight_init,
                         flg_train_weight=flg_train_weight, flg_bias=flg_bias, bias_init=bias_init, flg_train_bias=flg_train_bias,
                         flg_squash=flg_squash, u_max=u_max, flg_drop=flg_drop, dtype=dtype, device=device)
        self.target_traj = torch.as_tensor(target_traj, dtype=dtype, device=device).contiguous()

    def _raw_state_dim(self):
        return self.state_dim // 2

    def to(self, device):
        super().to(device)
        self.target_traj = self.target_traj.to(device)
