"""Autograd through the stand-alone class pieces: the policy module (CUDA vector-Jacobian product mcpilco_policy_backward), the GP
posterior w.r.t. its test inputs (GP_prior.get_estimate_from_alpha, Model_learning.get_next_state), and the reference's apply_policy
loop rebuilt from those pieces (MC_PILCO.py:615-674, :808-906) and differentiated by torch autograd."""
import types

import numpy as np
import pytest
import torch

import api_builders as AB
import helpers as Hh
import scenarios
from oracle import mcpilco_oracle as O

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import mcpilco_b200.model_learning.Model_learning as ML
    import mcpilco_b200.policy_learning.Cost_function as CF
    import mcpilco_b200.policy_learning.MC_PILCO as MCP
    import mcpilco_b200.policy_learning.Policy as PO
    return types.SimpleNamespace(ML=ML, CF=CF, MCP=MCP, PO=PO)


def relmax(a, b):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    b = b.detach().cpu().numpy() if hasattr(b, "detach") else np.asarray(b)
    return float(np.abs(a.reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-300))


def _scenario(name):
    return scenarios.ur5_full() if name == "ur5" else scenarios.scenario(name)


def _policy_case(name, nb, seed):
    """The scenario's policy with nb basis functions (fresh seeded centres / weights when nb differs): oracle dict (CPU, requires
    grad) and the McpPolicy the module would build."""
    from mcpilco_b200 import _pack as P
    sc = _scenario(name)
    p = dict(sc["policy"])
    rs = np.random.RandomState(seed)
    if nb != p["nb"]:
        c = p["centers"]
        p["centers"] = c[rs.randint(0, c.shape[0], nb)] + 0.3 * rs.randn(nb, c.shape[1])
        p["weight"] = rs.rand(sc["Du"], nb) - 0.5
        p["nb"] = nb
    sc["policy"] = p
    pol = Hh.oracle_policy(sc, requires_grad=True)
    Dp, Ds = p["centers"].shape[1], sc["Ds"]
    pst = P.policy_struct(p["kind"], nb, Dp, sc["Du"], Ds, u_max=p["u_max"], scale=p.get("scale"), angle=p.get("angle", ()),
                          non_angle=p.get("non_angle", ()), has_bias=p["bias"] is not None, use_drop=True)
    return sc, pol, pst


# (scenario, M, nb, p_dropout): every policy kind, bias + scale (delta), squash on (c*, ur5) and off (delta), injected masks with p > 0
# and p = 0, M in {0, 1, 2047, 2049, 65536}, nb in {1, 7, 33, 200, 512}, and the UR5-shaped policy (Dp = 24, Du = 6)
VJP_CASES = [("c1", 1, 1, 0.25), ("c2", 2047, 33, 0.0), ("c3", 2049, 7, 0.25), ("c4", 65536, 200, 0.25), ("delta", 0, 512, 0.1),
             ("delta", 2049, 512, 0.1), ("delta", 300, 12, 0.0), ("ur5", 2047, 200, 0.25)]


@pytest.mark.parametrize("name,M,nb,p", VJP_CASES)
def test_policy_vjp_matches_oracle_autograd(R, name, M, nb, p):
    """torch.ops.mcpilco.policy_forward + autograd (backward: the CUDA VJP) against autograd through O.policy_apply on the CPU, for
    log_ls, centers, W, bias and x.  Measured on a B200 (1000 W): at most 2.7e-15 relative max error over these cases."""
    from mcpilco_b200 import torch_ops as TO
    sc, pol, pst = _policy_case(name, nb, seed=M + nb)
    rs = np.random.RandomState(7)
    t = 1
    x = torch.tensor(rs.uniform(-1.5, 1.5, (M, sc["Ds"])), dtype=torch.float64)
    if sc["policy"]["kind"] == "target":
        x = x * 0.3 + Hh.T(sc["policy"]["target_traj"][t])
    G = torch.tensor(rs.randn(M, sc["Du"]), dtype=torch.float64)
    mask = torch.tensor((rs.rand(M, nb) >= p).astype(np.float64)) if p > 0 else None
    xr = x.clone().requires_grad_(True)
    u_ref = O.policy_apply(pol, xr, t, mask, p)
    names = [k for k in ("log_ls", "centers", "W", "bias") if pol[k] is not None]
    ref = torch.autograd.grad((u_ref * G).sum(), [pol[k] for k in names] + [xr], allow_unused=True)
    dp = {k: pol[k].detach().to(DEV).requires_grad_(True) for k in names}
    xd = x.to(DEV).requires_grad_(True)
    traj = pol.get("target_traj")
    u = torch.ops.mcpilco.policy_forward(TO.policy_tensor(pst), dp["log_ls"], dp["centers"], dp["W"], dp.get("bias"),
                                         None if traj is None else traj.to(DEV), xd, t, float(p),
                                         None if mask is None else mask.to(DEV, torch.uint8), 0, 0)
    assert u.shape == (M, sc["Du"]) and relmax(u, u_ref) < 1e-12 if M else u.shape == (0, sc["Du"])
    got = torch.autograd.grad((u * G.to(DEV)).sum(), [dp[k] for k in names] + [xd], allow_unused=True)
    for k, a, b in zip(names + ["x"], got, ref):
        b = torch.zeros_like(pol[k] if k != "x" else x) if b is None else b
        assert a is not None and a.shape == b.shape, k
        if M == 0:
            assert not a.any(), k
        else:
            assert relmax(a, b) < 1e-10, (k, relmax(a, b))


def test_policy_philox_dropout_finite_differences_and_determinism(R):
    """Class-level pol(x, t, p_dropout=0.25) with its Philox mask (seed from torch's RNG): the backward against central differences
    of the device forward with the same seed, on a sample of parameter and state entries; two backward calls are bit-identical.
    Measured on a B200 (1000 W): |fd - grad| at most 7e-11 of max(1, max |grad|) (6e-9 of the entry itself)."""
    sc = scenarios.scenario("c1")
    pol = AB.build_policy(R, sc, DEV)
    rs = np.random.RandomState(3)
    M = 3000
    x = torch.tensor(rs.uniform(-2, 2, (M, sc["Ds"])), dtype=torch.float64, device=DEV).requires_grad_(True)
    G = torch.tensor(rs.randn(M, sc["Du"]), dtype=torch.float64, device=DEV)
    params = [pol.log_lengthscales, pol.centers, pol.f_linear.weight]

    def loss():
        torch.manual_seed(11)
        return (pol(x, t=2, p_dropout=0.25) * G).sum()

    grads = [torch.autograd.grad(loss(), params + [x]) for _ in range(2)]
    for a, b in zip(*grads):
        assert torch.equal(a, b)
    g = grads[0]
    # the mask is not trivial: some units dropped, the rest kept
    torch.manual_seed(11)
    with torch.no_grad():
        u_drop = pol(x, t=2, p_dropout=0.25)
        u_keep = pol(x, t=2, p_dropout=0.0)
    assert not torch.equal(u_drop, u_keep)
    h = 1e-5
    for k, tensor in enumerate(params + [x]):
        flat = tensor.data.view(-1)
        for i in rs.choice(flat.numel(), 4, replace=False):
            old = float(flat[i])
            with torch.no_grad():
                flat[i] = old + h
                lp = float(loss())
                flat[i] = old - h
                lm = float(loss())
                flat[i] = old
            fd = (lp - lm) / (2 * h)
            an = float(g[k].view(-1)[i])
            assert abs(fd - an) <= 1e-6 * max(1.0, float(g[k].abs().max())), (k, int(i), fd, an)
    with pytest.raises(RuntimeError, match="double backward"):
        torch.autograd.grad(loss(), [pol.centers], create_graph=True)


@pytest.mark.parametrize("name", scenarios.ALL)
@pytest.mark.parametrize("linv", [True, False])
def test_posterior_vjp(R, name, linv):
    """get_estimate_from_alpha (both call forms) and get_next_state gradients w.r.t. their inputs against oracle autograd, with and
    without the triangular factor attached to K_X_inv.  Measured on a B200 (1000 W): mean 2.1e-14, var 1.9e-12; next state 1.7e-12,
    its gradients 4.2e-13 (state) and 3.9e-12 (input)."""
    import torch.distributions.normal as nrm
    from mcpilco_b200 import _ops as ops
    sc, g = scenarios.scenario(name), Hh.load_golden(name)
    T = AB.tensor_factory(DEV)
    ml = AB.build_model(R, sc, DEV)
    X = Hh.T(sc["X"])
    rs = np.random.RandomState(5)
    Gm, Gv = rs.randn(g["Xs"].shape[0], 1), rs.randn(g["Xs"].shape[0])
    for e, (gp, sp) in enumerate(zip(ml.gp_list, Hh.oracle_specs(sc))):
        Kinv = ml.K_X_inv_list[e] if linv else ml.K_X_inv_list[e].clone()
        assert (ops.attached_linv(Kinv) is not None) == linv
        xs = T(g["Xs"]).requires_grad_(True)
        mu, var = gp.get_estimate_from_alpha(ml.gp_inputs_tr_list[e], xs, ml.alpha_list[e], ml.m_X_list[e], Kinv)
        mu_only = gp.get_estimate_from_alpha(ml.gp_inputs_tr_list[e], xs, ml.alpha_list[e], ml.m_X_list[e])
        assert mu.requires_grad and var.requires_grad and mu_only.requires_grad
        gm, = torch.autograd.grad((mu * T(Gm)).sum(), xs, retain_graph=True)
        gv, = torch.autograd.grad((var * T(Gv)).sum(), xs)
        gm2, = torch.autograd.grad((mu_only * T(Gm)).sum(), xs)
        xr = Hh.T(g["Xs"]).requires_grad_(True)
        mr, vr = O.gp_predict(sp, X, ml.alpha_list[e].cpu(), ml.K_X_inv_list[e].cpu(), xr)
        rgm, = torch.autograd.grad((mr * Hh.T(Gm)).sum(), xr, retain_graph=True)
        rgv, = torch.autograd.grad((vr * Hh.T(Gv)).sum(), xr)
        assert relmax(gm, rgm) < 1e-9 and relmax(gm2, rgm) < 1e-9
        assert relmax(gv, rgv) < 1e-7
    # one model step through get_next_state, the reparameterisation noise injected as test_gpu_api.test_one_step does
    x0, u0 = Hh.T(g["states"][0]), Hh.T(g["inputs"][0])
    gps = [(sp, X, ml.alpha_list[e].cpu(), ml.K_X_inv_list[e].cpu()) for e, sp in enumerate(Hh.oracle_specs(sc))]
    xr, ur = x0.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    nxt_r, _, _ = O.next_state(Hh.oracle_model(sc), gps, xr, ur, Hh.T(sc["eps"][0]))
    W = Hh.T(rs.randn(*nxt_r.shape))
    rgx, rgu = torch.autograd.grad((nxt_r * W).sum(), [xr, ur])
    xd, ud = T(g["states"][0]).requires_grad_(True), T(g["inputs"][0]).requires_grad_(True)
    old = nrm._standard_normal
    nrm._standard_normal = lambda shape, dtype, device: T(sc["eps"][0])
    try:
        nxt, _, _ = ml.get_next_state(xd, ud)
    finally:
        nrm._standard_normal = old
    gx, gu = torch.autograd.grad((nxt * W.to(DEV)).sum(), [xd, ud])
    assert relmax(nxt, nxt_r) < 1e-10 and relmax(gx, rgx) < 1e-7 and relmax(gu, rgu) < 1e-7


@pytest.mark.parametrize("name", ["c1", "c4", "delta"])
def test_no_grad_calls_are_todays_calls(R, name):
    """Under torch.no_grad() the class calls are the direct _ops calls: bit-equal outputs, the same native launch counts, no graph.
    With grad, outputs equal them to rounding."""
    from mcpilco_b200 import _ops as ops
    sc, g = scenarios.scenario(name), Hh.load_golden(name)
    T = AB.tensor_factory(DEV)
    pol = AB.build_policy(R, sc, DEV)
    x = T(g["states"][1])

    def counted(fn):
        c0 = ops.launch_count()
        out = fn()
        return out, ops.launch_count() - c0

    with torch.no_grad():
        torch.manual_seed(1)
        u, n1 = counted(lambda: pol(x, t=1, p_dropout=0.25))
        torch.manual_seed(1)
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        u_ref, n2 = counted(lambda: ops.policy_forward(pol.policy_struct(), pol.policy_tensors(), x, t=1, p_dropout=0.25, seed=seed))
    assert torch.equal(u, u_ref) and n1 == n2 and not u.requires_grad
    torch.manual_seed(1)
    assert relmax(pol(x, t=1, p_dropout=0.25), u_ref) < 1e-14

    ml = AB.build_model(R, sc, DEV)
    gp, Xtr, alpha, m_X, Kinv = ml.gp_list[0], ml.gp_inputs_tr_list[0], ml.alpha_list[0], ml.m_X_list[0], ml.K_X_inv_list[0]
    xs = T(g["Xs"]).requires_grad_(True)
    spec = gp.gp_spec(Xtr.shape[1])
    with torch.no_grad():
        (mu, var), n1 = counted(lambda: gp.get_estimate_from_alpha(Xtr, xs, alpha, m_X, Kinv))
        (mu_r, var_r), n2 = counted(lambda: ops.gp_predict([ops.FittedGp(spec, Xtr, alpha, Kinv)], xs))
        m2, n3 = counted(lambda: gp.get_estimate_from_alpha(Xtr, xs, alpha, m_X))
        m2_r, n4 = counted(lambda: gp.get_mean(xs) + ops.gp_covariance(spec, xs, Xtr) @ alpha.reshape(-1, 1))
    assert torch.equal(mu, mu_r) and torch.equal(var, var_r[:, 0]) and n1 == n2 and not mu.requires_grad and not var.requires_grad
    assert torch.equal(m2, m2_r) and n3 == n4 and not m2.requires_grad
    mu_g, var_g = gp.get_estimate_from_alpha(Xtr, xs, alpha, m_X, Kinv)
    assert relmax(mu_g, mu_r) < 1e-12 and relmax(var_g, var_r[:, 0]) < 1e-9
    assert relmax(gp.get_estimate_from_alpha(Xtr, xs, alpha, m_X), m2_r) < 1e-12


@pytest.mark.parametrize("name", scenarios.ALL)
def test_reference_apply_policy_loop_from_class_pieces(R, name):
    """The reference's apply_policy loop (oracle.rollout / rollout_4pms) written with the class pieces: torch.ops.mcpilco.policy_forward
    with the golden step masks, get_next_state with injected eps, the generic Expected_cost path, cost.backward().  The policy .grad
    against the golden vectors (as test_apply_policy_cost_backward) and against the fused apply_policy on the same noise.  Measured on
    a B200 (1000 W): at most 6.4e-12 against the golden vectors, 7.3e-12 against the fused rollout."""
    import torch.distributions.normal as nrm
    from mcpilco_b200 import torch_ops as TO
    sc, g = scenarios.scenario(name), Hh.load_golden(name)
    T = AB.tensor_factory(DEV)
    ml = AB.build_model(R, sc, DEV)
    pol = AB.build_policy(R, sc, DEV)
    cls, par = AB.cost_spec(R, sc, DEV)
    cost_obj = R.CF.Expected_cost(cls(**par).cost_function)
    pst = TO.policy_tensor(pol.policy_struct())
    tens = pol.policy_tensors()
    traj = tens["target_traj"]
    masks = T(sc["masks"]).to(torch.uint8)
    p = float(sc["p_dropout"])

    def policy(x, t):
        return torch.ops.mcpilco.policy_forward(pst, tens["log_ls"], tens["centers"], tens["W"], tens["bias"], traj, x, t, p, masks[t], 0, 0)

    def step(x, u, t):
        old = nrm._standard_normal
        nrm._standard_normal = lambda shape, dtype, device: T(sc["eps"][t])
        try:
            return ml.get_next_state(x, u)[0]
        finally:
            nrm._standard_normal = old

    x0 = T(sc["x0_mean"]).reshape(1, -1) + T(sc["x0_var"]).sqrt().reshape(1, -1) * T(sc["eps0"])
    xs, us = [x0], [policy(x0, 0)]
    if "pms" in sc:
        q = sc["pms"]
        b, a = O.butter1(q["fc"])
        pos, vel, std = q["pos_idx"], q["vel_idx"], T(q["std_pos"])
        noisy, meas = [x0.clone()], [x0]
        for t in range(1, sc["H"]):
            nxt = step(xs[t - 1], us[t - 1], t - 1)
            xs.append(nxt)
            nz = nxt.clone()
            nz[:, pos] = nz[:, pos] + std * T(sc["meas_eps"][t - 1])
            nz[:, vel] = (nz[:, pos] - noisy[t - 1][:, pos]) / sc["model"]["T"]
            noisy.append(nz)
            ms = nz.clone()
            ms[:, vel] = (b[0] * nz[:, vel] + b[1] * noisy[t - 1][:, vel] - a[1] * meas[t - 1][:, vel]) / a[0]
            meas.append(ms)
            us.append(policy(ms, t))
    else:
        for t in range(1, sc["H"]):
            xs.append(step(xs[t - 1], us[t - 1], t - 1))
            us.append(policy(xs[t], t))
    states, inputs = torch.stack(xs), torch.stack(us)
    assert relmax(states, g["states"]) < 1e-5 and relmax(inputs, g["inputs"]) < 1e-5
    cost, _ = cost_obj(states, inputs, 0)
    cost.backward()
    params = {"g_log_ls": pol.log_lengthscales, "g_centers": pol.centers, "g_W": pol.f_linear.weight}
    if "g_bias" in g and pol.f_linear.bias.requires_grad:
        params["g_bias"] = pol.f_linear.bias
    for k, prm in params.items():
        assert prm.grad is not None and relmax(prm.grad, g[k]) < 1e-4, (k, relmax(prm.grad, g[k]))
    # the fused rollout on the same injected noise
    obj = AB.build_pilco(R, sc, ml, DEV)
    fused = obj.control_policy
    st, inp = obj.apply_policy(**AB.apply_kwargs(sc, DEV), _noise=dict(eps0=T(sc["eps0"]), eps=T(sc["eps"]), masks=T(sc["masks"]),
                                                                        **({"meas_eps": T(sc["meas_eps"])} if "pms" in sc else {})))
    obj.cost_function(st, inp, 0)[0].backward()
    fp = {"g_log_ls": fused.log_lengthscales, "g_centers": fused.centers, "g_W": fused.f_linear.weight, "g_bias": fused.f_linear.bias}
    for k, prm in params.items():
        assert relmax(prm.grad, fp[k].grad) < 1e-8, (k, relmax(prm.grad, fp[k].grad))
