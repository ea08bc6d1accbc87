"""INTEGRATION.md section 2 (method-level binding): the reference's own MC_PILCO class keeps the trial loop, data collection and
logging, and only the rollout methods are re-bound to mcpilco_b200's.  This CPU-collected test builds exactly that class — on a
stand-in with the reference's constructor (reference policy_learning/MC_PILCO.py:34-94), as the reference is not part of this
repository — and checks the wiring: every attribute the re-bound methods read exists on the
composed object, the objects they drive expose the hooks they call, and a call reaches the native layer (which refuses CPU tensors
loudly: there is no CPU fallback).  Runs in a subprocess so that the reference's top-level modules never enter the test process."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = textwrap.dedent(r'''
    import inspect, os, re, sys, types
    import numpy as np, torch
    ROOT = sys.argv[1]
    sys.path.insert(0, os.path.join(ROOT, "mc-pilco_b200"))

    class _Ref(torch.nn.Module):                           # stand-in with the reference's constructor (MC_PILCO.py:34-94)
        def __init__(self, T_sampling, state_dim, input_dim, f_sim, f_model_learning, model_learning_par, f_rand_exploration_policy,
                     rand_exploration_policy_par, f_control_policy, control_policy_par, f_cost_function, cost_function_par,
                     std_meas_noise=None, log_path=None, dtype=torch.float64, device=torch.device("cpu")):
            super().__init__()
            self.T_sampling, self.dtype, self.device, self.state_dim, self.input_dim = T_sampling, dtype, device, state_dim, input_dim
            self.std_meas_noise = np.zeros(state_dim) if std_meas_noise is None else std_meas_noise
            self.model_learning = f_model_learning(**model_learning_par)
            self.rand_exploration_policy = f_rand_exploration_policy(**rand_exploration_policy_par)
            self.control_policy = f_control_policy(**control_policy_par)
            self.cost_function = f_cost_function(**cost_function_par)
            self.state_samples_history, self.input_samples_history, self.noiseless_states_history = [], [], []
            self.num_data_collection, self.log_path = 0, log_path
    REF = types.SimpleNamespace(MC_PILCO=_Ref)
    import mcpilco_b200.policy_learning.MC_PILCO as B200
    import mcpilco_b200.model_learning.Model_learning as ML
    import mcpilco_b200.policy_learning.Policy as PO
    import mcpilco_b200.policy_learning.Cost_function as CF

    class MC_PILCO(REF.MC_PILCO):                      # trial loop, data collection, logging: the reference's
        apply_policy = B200.MC_PILCO.apply_policy      # the particle rollout: one fused CUDA call, one autograd node
        _rollout_call = B200.MC_PILCO._rollout_call
        _next_seed = B200.MC_PILCO._next_seed
        _initial_particles = B200.MC_PILCO._initial_particles
        _meas_struct = B200.MC_PILCO._meas_struct
        _trial_index = None; _seed_base = None; _rollouts = 0

    dev = torch.device("cpu")
    D = 6
    rbf = dict(active_dims=np.arange(D), lengthscales_init=np.ones(D), flg_train_lengthscales=True, lambda_init=np.ones(1), flg_train_lambda=False,
               sigma_n_init=0.1 * np.ones(1), flg_train_sigma_n=True, mean_init=np.zeros(1), sigma_n_num=None, dtype=torch.float64, device=dev)
    obj = MC_PILCO(T_sampling=0.05, state_dim=4, input_dim=1, f_sim=None,
                   f_model_learning=ML.Speed_Model_learning_RBF_angle_state,
                   model_learning_par=dict(num_gp=2, init_dict_list=[rbf, rbf], T_sampling=0.05, angle_indeces=[2], not_angle_indeces=[0, 1, 3],
                                           vel_indeces=[1, 3], not_vel_indeces=[0, 2], device=dev),
                   f_rand_exploration_policy=lambda **k: None, rand_exploration_policy_par={},
                   f_control_policy=PO.Sum_of_gaussians_with_angles,
                   control_policy_par=dict(state_dim=4, input_dim=1, num_basis=8, angle_indices=[2], non_angle_indices=[0, 1, 3],
                                           lengthscales_init=np.ones(5), centers_init=np.zeros((8, 5)), weight_init=np.zeros((1, 8)),
                                           flg_squash=True, u_max=10.0, flg_drop=True, device=dev),
                   f_cost_function=CF.Cart_pole_cost,
                   cost_function_par=dict(target_state=torch.tensor([np.pi, 0.0]), lengthscales=torch.tensor([3.0, 1.0]), angle_index=2, pos_index=0),
                   device=dev)
    assert MC_PILCO.apply_policy is B200.MC_PILCO.apply_policy
    # every attribute the re-bound methods read through `self.` exists on the composed object
    for fn in (B200.MC_PILCO.apply_policy, B200.MC_PILCO._rollout_call, B200.MC_PILCO._next_seed, B200.MC_PILCO._initial_particles,
               B200.MC_PILCO._meas_struct):
        for name in set(re.findall(r"\bself\.(\w+)", inspect.getsource(fn))):
            assert hasattr(obj, name), (fn.__name__, name)
    # ... and the objects they drive expose the hooks they call
    assert all(hasattr(obj.model_learning, h) for h in ("fitted_gps", "rollout_model_struct"))
    assert all(hasattr(obj.control_policy, h) for h in ("policy_struct", "policy_tensors", "flg_bias", "log_lengthscales", "centers", "f_linear"))
    assert hasattr(obj.cost_function, "fused_spec") and obj.cost_function.fused_spec(4, 5, None) is not None
    # a call reaches this repository's layer and fails loudly without a fitted model / CUDA tensors: no silent CPU path
    try:
        obj.apply_policy(np.zeros(4), 1e-4 * np.ones(4), False, None, None, False, 8, 5, p_dropout=0.1)
    except RuntimeError as e:
        assert "pre-trained" in str(e) or "no CPU fallback" in str(e) or "CUDA" in str(e), str(e)
    else:
        raise AssertionError("apply_policy on CPU tensors must raise")
    print("BINDING_OK")
''')


def test_method_level_binding_of_integration_md():
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "BINDING_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_integration_md_lists_the_rebound_methods():
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    for name in ("apply_policy", "_rollout_call", "_next_seed", "_initial_particles", "_meas_struct"):
        assert name in doc, name
