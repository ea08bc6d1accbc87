"""Dynamics-model objects — the reference's `model_learning/Model_learning.py` surface for the rollout hot path.

Same classes, constructor arguments and public state as the reference (Model_learning :43-493 and the RBF / angle-state /
speed-integration subclasses :496-760): `gp_list`, `gp_inputs`, `gp_output_list`, `alpha_list`, `m_X_list`, `K_X_inv_list`,
`gp_inputs_tr_list`, `norm_list`, `num_gp`.  `pretrain_gp` is the per-model-update precompute and `get_next_state` the
one-step prediction; both run in libmcpilco_b200.so.  The particle rollout does not call `get_next_state` step by step:
`MC_PILCO.apply_policy` hands `fitted_gps()` and `rollout_model_struct()` to the fused rollout.

`reinforce_model` / `train_gp_likelihood` (SURVEY.md §8f-2) train the hyper-parameters on the marginal likelihood with an analytic
gradient (one native call per epoch) instead of autograd through a Cholesky.  Out of scope (SURVEY.md §2 row 6): the SOR / L1
estimate paths, `SP_Speed_Model_learning_Furuta`.
"""
import torch
from torch.distributions.normal import Normal

from .. import _ops as ops
from .. import _pack as P
from ..gpr_lib.GP_prior import GP_prior as GP
from ..gpr_lib.GP_prior import Sparse_GP
from ..gpr_lib.GP_prior import Stationary_GP as SGP


class Model_learning(torch.nn.Module):
    """Training set + one GP per output (reference :43-493)."""

    _model_kind = "delta"

    def __init__(self, num_gp, init_dict_list, approximation_mode=None, approximation_dict=None, dtype=torch.float64,
                 device=torch.device("cpu"), flg_norm=False):
        super().__init__()
        self.num_samples = 0
        self.dtype, self.device = dtype, device
        self.init_dict_list = init_dict_list
        self.num_gp = num_gp
        self.alpha_list = [None] * num_gp
        self.m_X_list = [None] * num_gp
        self.K_X_inv_list = [None] * num_gp
        self.gp_inputs_tr_list = [None] * num_gp
        self.approximation_mode = approximation_mode
        if approximation_mode is None:
            self.get_gp_estimate = self.get_exact_gp_estimate
        elif approximation_mode == "SOD":
            self.approximation_dict = approximation_dict
            self.SOD_indices = [None] * num_gp
            self.get_gp_estimate = self.get_SOD_gp_estimate
            self.SOD_threshold_mode = approximation_dict["SOD_threshold_mode"]
            self.SOD_threshold = approximation_dict["SOD_threshold"]
            self.flg_SOD_permutation = approximation_dict["flg_SOD_permutation"]
        else:
            raise NotImplementedError("approximation_mode %r is outside the rollout hot path (exact and 'SOD' are supported)" % approximation_mode)
        self.init_gp_models()
        self.flg_norm = flg_norm
        self.norm_list = [1.0] * self.num_gp
        self._fitted_cache = None

    def init_gp_models(self):
        self.gp_list = torch.nn.ModuleList([self.get_gp(gp_index=i, init_dict=self.init_dict_list[i]) for i in range(self.num_gp)])

    def set_eval_mode(self):
        for gp in self.gp_list:
            gp.set_eval_mode()

    def set_training_mode(self):
        for gp in self.gp_list:
            gp.set_training_mode()

    def to(self, device):
        super().to(device)
        self.device = device
        for gp in self.gp_list:
            gp.to(device)

    def print_model(self):
        for i, gp in enumerate(self.gp_list):
            print("GP " + str(i) + ":")
            gp.print_model()

    # ---- data ------------------------------------------------------------------------------------------------------
    def add_data(self, new_state_samples, new_input_samples):
        """Append one trajectory's transitions to the GP training set (reference :123-147)."""
        st = torch.as_tensor(new_state_samples, dtype=self.dtype, device=self.device)
        inp = torch.as_tensor(new_input_samples, dtype=self.dtype, device=self.device)
        gp_in, gp_out = self.data_to_gp_IO(st, inp)
        if self.num_samples == 0:
            self.dim_state, self.dim_input = st.shape[1], inp.shape[1]
            self.gp_inputs, self.gp_output_list = gp_in, gp_out
            self.num_samples = st.shape[0]
        else:
            self.gp_inputs = torch.cat([self.gp_inputs, gp_in])
            self.gp_output_list = [torch.cat([self.gp_output_list[i], gp_out[i]], 0) for i in range(self.num_gp)]
            self.num_samples = self.gp_inputs.shape[0]

    def data_to_gp_input(self, states, inputs):
        return torch.cat([states, inputs], 1)

    def data_to_gp_output(self, states):
        return [(states[1:, i] - states[:-1, i]).reshape([-1, 1]) for i in range(self.dim_state)]

    def data_to_gp_IO(self, states, inputs):
        if not hasattr(self, "dim_state"):
            self.dim_state = states.shape[1]
        return self.data_to_gp_input(states, inputs)[:-1, :], self.data_to_gp_output(states)

    # ---- precompute --------------------------------------------------------------------------------------------------
    def pretrain_gp(self, gp_index):
        """alpha, m_X, K_X^-1 (and, in SOD mode, the greedy subset) of one GP (reference :163-208)."""
        gp = self.gp_list[gp_index]
        X, Y = self.gp_inputs, self.gp_output_list[gp_index]
        if self.approximation_mode == "SOD":
            if self.SOD_threshold_mode == "relative":
                threshold = self.SOD_threshold * torch.sqrt(gp.get_sigma_n_2())
            else:
                threshold = self.SOD_threshold[gp_index]
            self.SOD_indices[gp_index] = gp.get_SOD(X=X, Y=Y, threshold=threshold, flg_permutation=self.flg_SOD_permutation)
            idx = torch.as_tensor(self.SOD_indices[gp_index], device=X.device)
            X_tr, Y_tr = X[idx, :].contiguous(), Y[idx, :].contiguous()
        else:
            X_tr, Y_tr = X, Y
        Y_hat, var, alpha, m_X, K_X_inv = gp.get_estimate(X=X_tr, Y=Y_tr, X_test=X, flg_return_K_X_inv=True)
        self.K_X_inv_list[gp_index], self.alpha_list[gp_index] = K_X_inv, alpha
        self.m_X_list[gp_index], self.gp_inputs_tr_list[gp_index] = m_X, X_tr
        self._fitted_cache = None
        print("MSE gp " + str(gp_index) + ": ", torch.mean((Y - Y_hat) ** 2))

    def reinforce_model(self, optimization_opt_list=None):
        """Re-initialise the GPs, train each one's hyper-parameters, then precompute it (reference :149-161)."""
        self.init_gp_models()
        for gp_index in range(self.num_gp):
            self.train_gp(gp_index=gp_index, optimization_opt_dict=optimization_opt_list[gp_index])
            with torch.no_grad():
                self.pretrain_gp(gp_index=gp_index)

    def train_gp(self, gp_index, optimization_opt_dict):
        self.train_gp_likelihood(gp_index, optimization_opt_dict)

    def train_gp_likelihood(self, gp_index, optimization_opt_dict):
        """Full-batch optimisation of one GP's marginal likelihood (reference :398-421); `f_optimizer` is the reference's
        eval'd string, `criterion` the (mirrored) Marginal_log_likelihood class."""
        if self.flg_norm:
            self.norm_list[gp_index] = torch.max(torch.abs(self.gp_output_list[gp_index]))
        batch = [(self.gp_inputs, self.gp_output_list[gp_index] / self.norm_list[gp_index])]  # one batch = the whole training set
        f_optim = eval(optimization_opt_dict["f_optimizer"])
        gp = self.gp_list[gp_index]
        gp.fit_model(trainloader=batch, optimizer=f_optim(gp.parameters()), criterion=optimization_opt_dict["criterion"](),
                     N_epoch=optimization_opt_dict["N_epoch"], N_epoch_print=optimization_opt_dict["N_epoch_print"])

    def train_SOR_gp_likelihood(self, gp_index, optimization_opt_dict):
        raise NotImplementedError("subset-of-regressors training is outside the rollout hot path (and broken upstream)")

    # ---- what the fused rollout consumes -----------------------------------------------------------------------------
    def fitted_gps(self):
        """[ops.FittedGp] for all outputs; rebuilt when pretrain_gp ran or a list entry was replaced (load_model_from_log)."""
        def tkey(t):
            return None if t is None else (id(t), t._version, t.data_ptr(), tuple(t.shape))
        key = tuple((tkey(a), tkey(k), tkey(x), float(n), tuple(tkey(p) for p in gp.parameters()))
                    for a, k, x, n, gp in zip(self.alpha_list, self.K_X_inv_list, self.gp_inputs_tr_list, self.norm_list, self.gp_list))
        if self._fitted_cache is None or self._fitted_cache[0] != key:
            gps = []
            for i in range(self.num_gp):
                if self.alpha_list[i] is None:
                    raise RuntimeError("GP %d has not been pre-trained: call pretrain_gp(%d) first" % (i, i))
                X = self.gp_inputs_tr_list[i]
                gps.append(ops.FittedGp(self.gp_list[i].gp_spec(X.shape[1]), X, self.alpha_list[i], self.K_X_inv_list[i],
                                        var_scale=float(self.norm_list[i]) ** 2))
            # the keyed tensors are held (FittedGp keeps Xtr / alpha / Kinv views alive), so an id cannot be recycled under the cache
            self._fitted_cache = (key, gps, (list(self.alpha_list), list(self.K_X_inv_list), list(self.gp_inputs_tr_list)))
        return self._fitted_cache[1]

    def rollout_model_struct(self, Ds, Du, particle_pred=True):
        return P.model_struct("delta", Ds, Du, self.num_gp, use_trig=False, particle_pred=particle_pred)

    # ---- one-step prediction -----------------------------------------------------------------------------------------
    def get_exact_gp_estimate(self, gp_inputs, gp_index_list=None):
        """Posterior mean / variance lists at gp_inputs (reference :265-289); one native call for all outputs.  Differentiable (once)
        w.r.t. gp_inputs; the fitted GPs (alpha, K_X_inv, training inputs, hyper-parameters) receive no gradient."""
        idx = list(range(self.num_gp)) if gp_index_list is None else list(gp_index_list)
        fitted = self.fitted_gps()
        mean, var = ops.gp_predict([fitted[i] for i in idx], gp_inputs)
        # fitted_gps() folds norm**2 into the variance; the reference applies it in get_next_state, after this call
        mean_list = [mean[:, k:k + 1] for k in range(len(idx))]
        var_list = [(var[:, k:k + 1] / float(self.norm_list[i]) ** 2) for k, i in enumerate(idx)]
        return mean_list, var_list

    def get_SOD_gp_estimate(self, gp_inputs, gp_index_list):
        return self.get_exact_gp_estimate(gp_inputs, gp_index_list)

    def get_one_step_gp_out(self, states, inputs):
        gp_inputs = self.data_to_gp_input(states=states, inputs=inputs)
        mean_list, var_list = self.get_gp_estimate(gp_inputs=gp_inputs, gp_index_list=range(self.num_gp))
        return gp_inputs, None, mean_list, var_list

    def get_gp_estimate_from_data(self, states, inputs, flg_pretrain=False, gp_index_list=None, flg_onestep=False):
        idx = range(self.num_gp) if gp_index_list is None else gp_index_list
        if flg_onestep:
            gp_inputs, gp_outputs_list = self.data_to_gp_input(states=states, inputs=inputs), None
        else:
            gp_inputs, gp_outputs_list = self.data_to_gp_IO(states=states, inputs=inputs)
        if flg_pretrain:
            for i in idx:
                self.pretrain_gp(gp_index=i)
        mean_list, var_list = self.get_gp_estimate(gp_inputs=gp_inputs, gp_index_list=idx)
        return gp_inputs, gp_outputs_list, mean_list, var_list

    def get_next_state(self, current_state, current_input, particle_pred=True):
        """One model step for a batch of states (reference :210-229): variance scaled by norm**2, the mean is not.  Differentiable
        (once) w.r.t. current_state and current_input; the GPs receive no gradient."""
        _, _, mean_list, var_list = self.get_one_step_gp_out(states=current_state, inputs=current_input)
        var_list = [v * self.norm_list[i] ** 2 for i, v in enumerate(var_list)]
        return self.get_next_state_from_gp_output(current_state=current_state, current_input=current_input, gp_output_mean_list=mean_list,
                                                  gp_output_var_list=var_list, particle_pred=particle_pred)

    def _sample_delta(self, mean_list, var_list, particle_pred):
        mean, var = torch.cat(mean_list, 1), torch.cat(var_list, 1)
        return (Normal(mean, torch.sqrt(var)).rsample() if particle_pred else mean), mean, var

    def get_next_state_from_gp_output(self, current_state, current_input, gp_output_mean_list, gp_output_var_list, particle_pred=True):
        """x' = x + delta (reference :471-493)."""
        delta, mean, var = self._sample_delta(gp_output_mean_list, gp_output_var_list, particle_pred)
        return current_state + delta, mean, var

    def get_gp(self, gp_index, init_dict):
        raise NotImplementedError()


class Model_learning_RBF(Model_learning):
    """Every output is an RBF GP (reference :496-525)."""

    def get_gp(self, gp_index, init_dict):
        return SGP.RBF(**init_dict)


class Model_learning_RBF_angle_state(Model_learning):
    """RBF GPs on the sin/cos-extended state (reference :528-579)."""

    def __init__(self, num_gp, init_dict_list, angle_indeces, not_angle_indeces, approximation_mode=None, approximation_dict=None,
                 dtype=torch.float64, device=torch.device("cpu"), flg_norm=False):
        self.angle_indeces, self.not_angle_indeces = angle_indeces, not_angle_indeces
        super().__init__(num_gp=num_gp, init_dict_list=init_dict_list, approximation_mode=approximation_mode,
                         approximation_dict=approximation_dict, dtype=dtype, device=device, flg_norm=flg_norm)

    def get_gp(self, gp_index, init_dict):
        return SGP.RBF(**init_dict)

    def data_to_gp_input(self, states, inputs):
        """[x[not_angle], sin x[angle], cos x[angle], u]."""
        return torch.cat([states[:, self.not_angle_indeces], torch.sin(states[:, self.angle_indeces]),
                          torch.cos(states[:, self.angle_indeces]), inputs], 1)

    def rollout_model_struct(self, Ds, Du, particle_pred=True):
        return P.model_struct("delta", Ds, Du, self.num_gp, angle=self.angle_indeces, not_angle=self.not_angle_indeces, use_trig=True,
                              particle_pred=particle_pred)


class Model_learning_RBF_MPK_angle_state(Model_learning_RBF_angle_state):
    """RBF + Volterra-MPK GPs on the sin/cos-extended state (reference :582-616)."""

    def get_gp(self, gp_index, init_dict):
        return GP.Sum_Independent_GP(SGP.RBF(**init_dict[0]), Sparse_GP.get_Volterra_MPK_GP(**init_dict[1]))


class Speed_Model_learning_RBF_angle_state(Model_learning):
    """GPs predict velocity changes; positions are integrated (reference :619-718).  vel_indeces[k] is the derivative of
    not_vel_indeces[k]."""

    def __init__(self, num_gp, init_dict_list, T_sampling, angle_indeces, not_angle_indeces, vel_indeces, not_vel_indeces,
                 approximation_mode=None, approximation_dict=None, dtype=torch.float64, device=torch.device("cpu"), flg_norm=False):
        self.vel_indeces, self.not_vel_indeces = vel_indeces, not_vel_indeces
        self.angle_indeces, self.not_angle_indeces = angle_indeces, not_angle_indeces
        self.T_sampling = T_sampling
        super().__init__(num_gp=num_gp, init_dict_list=init_dict_list, approximation_mode=approximation_mode,
                         approximation_dict=approximation_dict, dtype=dtype, device=device, flg_norm=flg_norm)

    def get_gp(self, gp_index, init_dict):
        return SGP.RBF(**init_dict)

    def data_to_gp_output(self, states):
        return [(states[1:, i] - states[:-1, i]).reshape([-1, 1]) for i in self.vel_indeces]

    def data_to_gp_input(self, states, inputs):
        return torch.cat([states[:, self.not_angle_indeces], torch.sin(states[:, self.angle_indeces]),
                          torch.cos(states[:, self.angle_indeces]), inputs], 1)

    def get_next_state_from_gp_output(self, current_state, current_input, gp_output_mean_list, gp_output_var_list, particle_pred=True):
        """vel' = vel + delta ; pos' = pos + T vel + T/2 delta (reference :685-718)."""
        delta, mean, var = self._sample_delta(gp_output_mean_list, gp_output_var_list, particle_pred)
        nxt = torch.zeros_like(current_state)
        nxt[:, self.vel_indeces] = current_state[:, self.vel_indeces] + delta
        nxt[:, self.not_vel_indeces] = (current_state[:, self.not_vel_indeces] + self.T_sampling * current_state[:, self.vel_indeces]
                                        + self.T_sampling / 2 * delta)
        return nxt, mean, var

    def rollout_model_struct(self, Ds, Du, particle_pred=True):
        return P.model_struct("speed", Ds, Du, self.num_gp, angle=self.angle_indeces, not_angle=self.not_angle_indeces,
                              vel=self.vel_indeces, pos=self.not_vel_indeces, T=self.T_sampling, use_trig=True, particle_pred=particle_pred)


class Speed_Model_learning_RBF_MPK_angle_state(Speed_Model_learning_RBF_angle_state):
    """Speed-integration model with RBF + Volterra-MPK GPs (reference :721-760)."""

    def get_gp(self, gp_index, init_dict):
        return GP.Sum_Independent_GP(SGP.RBF(**init_dict[0]), Sparse_GP.get_Volterra_MPK_GP(**init_dict[1]))
