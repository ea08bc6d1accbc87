"""GP fitting beyond one 64-point block: the precompute factors (blocked Cholesky, L^-1, K^-1, alpha) and the NLML value and
gradient against fp64 references on the CPU, at sizes chosen from the dispatch rules of the precompute's update products.

The NLML reference works in FIELD space: it builds K from the very McpGpSpec fields the kernels receive,

    K = lambda exp(-sum_j ((x_j - x'_j) inv_ls_j)^2) [has_se] + sum_p prod_{f < deg_p} (sum_j w2[p][f][j] x_j x'_j + w2[p][f][MAX_D])
        + sigma_n2 I,

takes  NLML = 0.5 (r^T K^-1 r + log det K),  r = y - mean0,  through torch.linalg.cholesky / cholesky_solve (no explicit inverse, so
it shares no algorithm with the device), and differentiates it with autograd w.r.t. the fields.  Its own correctness is checked on
the CPU (tests without the gpu mark): K against the oracle's covariance, the gradient against central differences of its value.

Precompute sizes (np = N rounded up to 64-point blocks, split nb/2 | nb - nb/2 at every level of the recursion):
  129, 191 -> 3 blocks, uneven 1|2 split, 32 x 32 tiles;  300, 400 -> 5, 7 blocks;  1300 -> 21 blocks, 64 x 64 tiles, final W W^T on
  the TMA kernel with a half tile (1344 = 10.5 * 128);  1472 -> final product with a half tile;  2880, 3008, 4160 -> top-level
  updates on the TMA kernel with M or N = 64 mod 128 and an uneven split.  test_sizes_reach_intended_kernels pins this table to
  the launched kernels, so a later change of a dispatch threshold shows up as a failure instead of silently emptying these tests.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mcpilco_b200 import _native as Nat
from mcpilco_b200 import _ops as ops
from mcpilco_b200 import _pack as P
from mcpilco_b200 import workloads as W
from oracle import mcpilco_oracle as O

F64 = torch.float64
U = 2.0 ** -53
GRAD_SIZE = 4 + Nat.MAX_D + Nat.MAX_POLY * Nat.MAX_DEG * (Nat.MAX_D + 1)   # mcpilco_gp_nlml_grad_size()


# ---------------------------------------------------------------------------------------------------------------------------------
# field-space fp64 reference (CPU, torch)
# ---------------------------------------------------------------------------------------------------------------------------------
def field_slots(spec):
    """Every spec field the NLML gradient covers, as (device output index, field path), in the order of the reference's theta:
    lambda, mean0, sigma_n2, inv_ls[0..D), then per term p and factor f < deg_p: w2[p][f][0..D), offset w2[p][f][MAX_D]."""
    D = spec.D
    out = [(ops.NLML_LAMBDA, ("lambda_",)), (ops.NLML_MEAN, ("mean0",)), (ops.NLML_SN2, ("sigma_n2",))]
    out += [(ops.NLML_ILS + j, ("inv_ls", j)) for j in range(D)]
    for p in range(spec.n_poly):
        for f in range(spec.poly_deg[p]):
            o = ops.nlml_poly_offset(p, f)
            out += [(o + j, ("poly_w2", p, f, j)) for j in range(D)] + [(o + Nat.MAX_D, ("poly_w2", p, f, Nat.MAX_D))]
    return out


def get_field(spec, path):
    v = getattr(spec, path[0])
    for i in path[1:]:
        v = v[i]
    return float(v)


def set_field(spec, path, value):
    if len(path) == 1:
        setattr(spec, path[0], value)
        return
    v = getattr(spec, path[0])
    for i in path[1:-1]:
        v = v[i]
    v[path[-1]] = value


def spec_theta(spec):
    return torch.tensor([get_field(spec, path) for _, path in field_slots(spec)], dtype=F64)


def field_K(spec, X, theta, noise=True):
    """K from the spec fields held in theta (layout of field_slots)."""
    N, D = X.shape
    lam, sn2, inv_ls = theta[0], theta[2], theta[3:3 + D]
    K = torch.zeros(N, N, dtype=F64)
    if spec.has_se:
        d2 = torch.zeros(N, N, dtype=F64)
        for j in range(D):
            d2 = d2 + ((X[:, j:j + 1] - X[:, j:j + 1].t()) * inv_ls[j]) ** 2
        K = lam * torch.exp(-d2)
    k = 3 + D
    for p in range(spec.n_poly):
        prod = torch.ones(N, N, dtype=F64)
        for f in range(spec.poly_deg[p]):
            w = theta[k:k + D + 1]
            prod = prod * ((X * w[:D]) @ X.t() + w[D])
            k += D + 1
        K = K + prod
    return K + sn2 * torch.eye(N, dtype=F64) if noise else K


def ref_nlml_value(spec, X, y, theta):
    L = torch.linalg.cholesky(field_K(spec, X, theta))
    r = (y.reshape(-1) - theta[1]).reshape(-1, 1)
    a = torch.cholesky_solve(r, L)
    return 0.5 * ((r * a).sum() + 2.0 * torch.log(torch.diagonal(L)).sum())


def ref_nlml(spec, X, y):
    """Value and field gradient in the device's output layout (numpy [GRAD_SIZE]); entries outside the spec stay zero."""
    X, y = X.detach().cpu(), y.detach().cpu()
    theta = spec_theta(spec).requires_grad_(True)
    v = ref_nlml_value(spec, X, y, theta)
    g, = torch.autograd.grad(v, theta)
    out = np.zeros(GRAD_SIZE)
    out[0] = float(v.detach())
    for (idx, _), gi in zip(field_slots(spec), g.numpy()):
        out[idx] = gi
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
# problems
# ---------------------------------------------------------------------------------------------------------------------------------
def well_spec(N, D, form, rs):
    """Kernels of a well-conditioned regime (cond(K) ~ 10 .. 10^2) for N inputs in [-1.5, 1.5]^D: lengthscales about half the input
    spread, polynomial weights ~ 1 / sqrt(N) (so that no term's largest eigenvalue grows with N), noise variance 0.12 .. 0.25.
    form: "se" | "se_mean" | "volterra" (SE + degrees 1, 2, 3) | "se_lin" (SE + degree 1, the UR5 kernel) | "mpk" (degrees 1 and 2,
    no SE term) | "c1" (SE + degrees 1, 2: the cart-pole kernel)."""
    n_deg = {"se": 0, "se_mean": 0, "volterra": 3, "se_lin": 1, "mpk": 2, "c1": 2}[form]
    mpk = [np.exp(0.2 * rs.randn((k + 1) * D + (1 if k == 0 else 0))) / np.sqrt(N) for k in range(n_deg)]
    d = {"D": D, "log_ls": None if form == "mpk" else np.log(0.5) + 0.2 * rs.randn(D), "lambda": 1.3,
         "mean": 0.0 if form in ("se", "c1") else -0.4, "mpk": mpk, "sigma_n": 0.35 + 0.15 * rs.rand()}
    s = P.spec_from_dict(d)
    if form == "mpk":
        s.mean0 = 0.25          # the field is honoured without an SE term as well
    return s


def well_problem(N, D, form, seed=0):
    rs = np.random.RandomState(1000 * D + N + seed)
    X = torch.tensor(rs.uniform(-1.5, 1.5, (N, D)), dtype=F64)
    y = torch.tensor(rs.randn(N), dtype=F64)
    return well_spec(N, D, form, rs), X, y


def cartpole_problem(N, seed=0):
    """C1 (SE + MPK(2)) on cart-pole transitions; sigma_n = e^-4.2 (C1's own) up to N = 400, 0.1 above so that K stays positive
    definite in fp64 (test_size_independent_properties_large does the same)."""
    sn = float(np.exp(-4.2)) if N <= 400 else 0.1
    X, Y = W.cartpole_transitions(N, sn, np.random.RandomState(N + seed))
    spec = P.spec_from_dict({"D": 6, "log_ls": W.SE_LOG_LS, "lambda": 1.0, "mean": 0.0, "mpk": [np.exp(W.MPK1_LOG), np.exp(W.MPK2_LOG)],
                             "sigma_n": sn})
    return spec, torch.tensor(X, dtype=F64), torch.tensor(Y[:, 0].copy(), dtype=F64)


def relmax(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def norm1(A):
    return float(torch.linalg.matrix_norm(A, ord=1))


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU self-checks of the reference
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_se", [True, False])
def test_reference_covariance_matches_oracle(with_se):
    """(a) field_K from the packed spec equals the oracle's covariance for the equivalent log-parameter spec (SE + Volterra terms of
    degree 1, 2 and 3; and the same without the SE term).  Measured: 8.9e-16 of max|K|."""
    rs = np.random.RandomState(5)
    D = 5
    log_ls = 0.3 * rs.randn(D) if with_se else None
    mpk_log = [np.log(0.2) + 0.3 * rs.randn((k + 1) * D + (1 if k == 0 else 0)) for k in range(3)]
    spec = P.spec_from_dict({"D": D, "log_ls": log_ls, "lambda": 1.7, "mean": 0.3, "mpk": [np.exp(m) for m in mpk_log], "sigma_n": 0.2})
    so = O.make_spec(D, log_ls=log_ls, log_lambda=np.log(1.7), mean=0.3, mpk_log_pars=mpk_log, sigma_n=0.2)
    X = torch.tensor(rs.uniform(-2, 2, (70, D)), dtype=F64)
    Ko = O.gp_cov(so, X, None, noise=True)
    K = field_K(spec, X, spec_theta(spec))
    assert spec.has_se == (1 if with_se else 0) and spec.n_poly == 3 and list(spec.poly_deg) == [1, 2, 3]
    assert float((K - Ko).abs().max()) <= 1e-14 * float(Ko.abs().max())


def test_reference_gradient_matches_central_differences():
    """(b) the autograd field gradient of the reference against central differences of its own value, every slot (mean0 included),
    and nothing written outside the spec's slots."""
    spec, X, y = well_problem(40, 4, "volterra")
    ref = ref_nlml(spec, X, y)
    slots = field_slots(spec)
    theta0 = spec_theta(spec)
    for k, (idx, path) in enumerate(slots):
        h = 1e-4 * max(abs(float(theta0[k])), 1e-3)
        tp, tm = theta0.clone(), theta0.clone()
        tp[k] += h
        tm[k] -= h
        fd = (float(ref_nlml_value(spec, X, y, tp)) - float(ref_nlml_value(spec, X, y, tm))) / (2 * h)
        assert abs(fd - ref[idx]) <= 1e-6 * abs(ref[idx]) + 1e-8, (path, fd, ref[idx])
    used = {0} | {idx for idx, _ in slots}
    assert all(ref[i] == 0.0 for i in range(GRAD_SIZE) if i not in used)


def test_well_conditioned_problems_are_well_conditioned():
    """The 'well-conditioned' regime of the GPU tests is what its name says (cond_2(K) <= 10^2), so that forward errors of 1e-13
    are the right yardstick there."""
    for N, D, form in [(300, 6, "c1"), (400, 24, "se_lin"), (257, 32, "volterra"), (300, 13, "mpk"), (1300, 10, "se_mean")]:
        spec, X, _ = well_problem(N, D, form)
        ev = torch.linalg.eigvalsh(field_K(spec, X, spec_theta(spec)))
        assert float(ev[-1] / ev[0]) < 1e2, (N, D, form, float(ev[-1] / ev[0]))


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
DEV = "cuda:0"


@pytest.fixture(scope="module")
def gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    assert Nat.lib().mcpilco_gp_nlml_grad_size() == GRAD_SIZE
    return torch.device(DEV)


def precompute_into_nan(spec, X, y):
    """mcpilco_gp_precompute with every output buffer pre-filled with NaN (ops.gp_precompute hands it zeroed buffers), returning the
    whole [N, ld] buffers of K^-1, L and L^-1: what the kernels leave in the padding columns [N, ld) is then visible."""
    n = X.shape[0]
    ld = ops.even_ld(n)
    L_ = ops._enter(X.device)
    nan = float("nan")
    alpha = torch.full((n,), nan, dtype=F64, device=X.device)
    Kb, Lb, Rb = (torch.full((n, ld), nan, dtype=F64, device=X.device) for _ in range(3))
    wsb = L_.mcpilco_gp_precompute_workspace_bytes(n)
    ws = torch.empty(wsb, dtype=torch.uint8, device=X.device)
    Nat.check(L_.mcpilco_gp_precompute(C.byref(spec), ops._ptr(X), ops._ptr(y), n, ops._ptr(alpha), ops._ptr(Kb), ld, ops._ptr(Lb),
                                       ops._ptr(Rb), ops._ptr(ws), wsb, ops._stream(X.device)))
    return alpha, Kb, Lb, Rb


PRE_N = [1, 2, 63, 64, 65, 127, 129, 191, 300, 400, 1300, 1472, 2880, 3008, 4160]
# bounds ~10x the maxima measured on a B200 (1000 W power limit) over all sizes and both regimes (see test_precompute_factors)
TOL_FWD = 5e-14             # forward errors (relmax) in the well-conditioned regime
C_CHOL, C_RL, C_KINV, C_ALPHA = 30.0, 0.75, 10.0, 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("regime", ["well", "cartpole"])
@pytest.mark.parametrize("N", PRE_N)
def test_precompute_factors(gpu, N, regime):
    """Blocked Cholesky L, R = L^-1, K^-1 = R^T R and alpha = K^-1 (y - mean0) at the dispatch-table sizes, D = 6, SE + MPK(2).

    Both regimes: backward errors, with u = 2^-53 and K = ops.gp_covariance(spec, X, None, add_noise=True),
        |L L^T - K| <= c (N+1) u |L||L|^T elementwise,   ||R L - I||_max <= c N u || |R||L| ||_max,
        ||K Kinv - I||_1 / (||K||_1 ||Kinv||_1) <= c N u,   |alpha - Kinv r| <= c N u |Kinv||r| elementwise (r = y - mean0);
    L and R exactly lower triangular with diag(L) > 0, Kinv exactly symmetric, the padding columns [N, ld) of Kinv and L^-1 exactly
    zero; alpha / Kinv bit-identical with and without the L / L^-1 exports; two identical calls bit-identical.
    Well-conditioned regime (cond_1(K) <= 10^2): in addition forward errors of L, R, Kinv and alpha against LAPACK (CPU) on the same K.

    Measured on a B200 (1000 W), maxima over the 15 sizes: c = 2.97 (L L^T; the well-conditioned regime, whose L21 = A21 L11^-T is
    formed with the explicit block inverse, 0.85 in the cart-pole one), 0.073 (R L), 1.0 (K Kinv, at N = 1; <= 0.81 from N = 2),
    0.051 (alpha); forward errors <= 5.2e-15 (alpha at N = 4160; L <= 1.4e-15, R <= 2.8e-15, Kinv <= 4.5e-15); cond_1(K) 1 .. 44
    (well-conditioned), up to 1.8e6 (cart-pole).
    """
    spec, X, y = well_problem(N, 6, "c1") if regime == "well" else cartpole_problem(N)
    Xg, yg = X.to(gpu), y.to(gpu)
    a0, K0 = ops.gp_precompute(spec, Xg, yg)
    alpha, Kb, Lb, Rb = precompute_into_nan(spec, Xg, yg)
    a2, Kb2, Lb2, Rb2 = precompute_into_nan(spec, Xg, yg)
    torch.cuda.synchronize()
    Kinv, L, R = Kb[:, :N], Lb[:, :N], Rb[:, :N]
    # determinism and independence of the optional exports
    assert torch.equal(alpha, a2) and torch.equal(Kb, Kb2) and torch.equal(Rb, Rb2) and torch.equal(L, Lb2[:, :N])
    assert torch.equal(a0.reshape(-1), alpha) and torch.equal(K0, Kinv)
    # structure and padding
    ld = ops.even_ld(N)
    assert K0.stride() == (ld, 1)
    assert torch.equal(K0.as_strided((N, ld), (ld, 1))[:, N:], torch.zeros(N, ld - N, dtype=F64, device=gpu))
    assert torch.equal(Kb[:, N:], torch.zeros(N, ld - N, dtype=F64, device=gpu))
    assert torch.equal(Rb[:, N:], torch.zeros(N, ld - N, dtype=F64, device=gpu))
    assert torch.equal(L, torch.tril(L)) and torch.equal(R, torch.tril(R)) and bool((torch.diagonal(L) > 0).all())
    assert torch.equal(Kinv, Kinv.t())
    # backward errors
    K = ops.gp_covariance(spec, Xg, None, add_noise=True)
    I = torch.eye(N, dtype=F64, device=gpu)
    aL, aR = L.abs(), R.abs()
    c_chol = float(((L @ L.t() - K).abs() / ((N + 1) * U * (aL @ aL.t()))).max())
    c_rl = float((R @ L - I).abs().max() / (N * U * float((aR @ aL).max())))
    c_kinv = norm1(K @ Kinv - I) / (norm1(K) * norm1(Kinv) * N * U)
    r = yg - spec.mean0
    c_alpha = float(((alpha - Kinv @ r).abs() / (N * U * (Kinv.abs() @ r.abs()))).max())
    cond = norm1(K) * norm1(Kinv)
    msg = "N=%5d %-8s cond_1 %.2e  c: chol %.3g  RL %.3g  KKinv %.3g  alpha %.3g" % (N, regime, cond, c_chol, c_rl, c_kinv, c_alpha)
    if regime == "well":
        Kc = K.cpu()
        Lr = torch.linalg.cholesky(Kc)
        Rr = torch.linalg.solve_triangular(Lr, torch.eye(N, dtype=F64), upper=False)
        fwd = {"L": relmax(L.cpu(), Lr), "R": relmax(R.cpu(), Rr), "Kinv": relmax(Kinv.cpu(), torch.cholesky_inverse(Lr)),
               "alpha": relmax(alpha.cpu(), torch.cholesky_solve((y - spec.mean0).reshape(-1, 1), Lr).reshape(-1))}
        msg += "  fwd: " + " ".join("%s %.2e" % kv for kv in fwd.items())
    print(msg)
    assert c_chol <= C_CHOL and c_rl <= C_RL and c_kinv <= C_KINV and c_alpha <= C_ALPHA, msg
    if regime == "well":
        assert cond <= 1e2, msg
        assert max(fwd.values()) <= TOL_FWD, msg


NLML_CASES = [  # (N, D, kernel form, regime): every N, every DT instantiation (4, 6, 8, 12, 16, 24, 32) and every kernel form
    (65, 3, "se", "well"),
    (65, 8, "mpk", "well"),
    (257, 5, "volterra", "well"),
    (257, 32, "volterra", "well"),
    (300, 13, "mpk", "well"),
    (300, 6, "c1", "cartpole"),
    (400, 24, "se_lin", "well"),
    (400, 6, "c1", "cartpole"),
    (1300, 10, "se_mean", "well"),
    (3008, 6, "c1", "cartpole"),
]
TOL_NLML_WELL = 1e-13       # measured: 1.3e-14 (d/dlambda, N = 65)
TOL_NLML_REAL = 1e-6        # the golden-file test's bound; its floor is about cond(K) u.  Measured: 3.6e-11 (d/dmean0, N = 3008)


def nlml_groups(spec):
    """Output entries compared together (relmax within a group): the value, lambda, mean0, sigma_n2, inv_ls[0..D), each (p, f) row."""
    D = spec.D
    g = {"nlml": [0], "lambda": [ops.NLML_LAMBDA], "mean0": [ops.NLML_MEAN], "sigma_n2": [ops.NLML_SN2],
         "inv_ls": list(range(ops.NLML_ILS, ops.NLML_ILS + D))}
    for p in range(spec.n_poly):
        for f in range(spec.poly_deg[p]):
            o = ops.nlml_poly_offset(p, f)
            g["w2[%d][%d]" % (p, f)] = list(range(o, o + D)) + [o + Nat.MAX_D]
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("N,D,form,regime", NLML_CASES)
def test_nlml_value_and_field_gradient(gpu, N, D, form, regime):
    """ops.gp_nlml (precompute + nlml_grad_kernel over a (cdiv(N,256), cdiv(N,64)) grid + fixed-order cross-block sums) against the
    field-space reference: every entry of the output, those outside the spec exactly zero."""
    spec, X, y = well_problem(N, D, form) if regime == "well" else cartpole_problem(N)
    out = ops.gp_nlml(spec, X.to(gpu), y.to(gpu)).cpu().numpy()
    ref = ref_nlml(spec, X, y)
    used = {0} | {idx for idx, _ in field_slots(spec)}
    outside = [i for i in range(GRAD_SIZE) if i not in used]
    assert all(out[i] == 0.0 for i in outside), [i for i in outside if out[i] != 0.0]
    errs = {k: relmax(out[ix], ref[ix]) for k, ix in nlml_groups(spec).items() if np.abs(ref[ix]).max() > 0}
    worst = max(errs, key=errs.get)
    print("N=%5d D=%2d %-8s %-8s nlml %.6e  worst %s %.2e" % (N, D, form, regime, ref[0], worst, errs[worst]))
    if not spec.has_se:
        assert out[ops.NLML_LAMBDA] == 0.0 and all(out[ops.NLML_ILS + j] == 0.0 for j in range(D))
    assert errs[worst] <= (TOL_NLML_WELL if regime == "well" else TOL_NLML_REAL), errs


@pytest.mark.gpu
def test_nlml_gradient_matches_central_differences_of_the_device_value(gpu):
    """Independent of the reference: at N = 300 (5 x 2 blocks of the gradient grid; 5 precompute leaves) the device gradient of every
    field against central differences of the device value."""
    spec, X, y = well_problem(300, 5, "volterra")
    Xg, yg = X.to(gpu), y.to(gpu)
    out = ops.gp_nlml(spec, Xg, yg).cpu().numpy()
    gmax = max(abs(out[idx]) for idx, _ in field_slots(spec))
    for idx, path in field_slots(spec):
        v0 = get_field(spec, path)
        h = 1e-4 * max(abs(v0), 1e-2)
        vals = []
        for s in (1, -1):
            sp = Nat.GpSpec.from_buffer_copy(spec)
            set_field(sp, path, v0 + s * h)
            vals.append(float(ops.gp_nlml(sp, Xg, yg)[0]))
        fd = (vals[0] - vals[1]) / (2 * h)
        assert abs(fd - out[idx]) <= 1e-5 * (abs(out[idx]) + 1e-3 * gmax), (path, fd, out[idx])   # reference: 6.5e-8


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["c1", "c2", "c4"])
def test_class_nlml_at_real_training_shapes(gpu, key):
    """Marginal_log_likelihood()(gp(X), Y).backward() at the reference's real training sizes (C1 / C2: N = 300, D = 6; C4: six GPs
    with D = 24 at N = 400), value and every trainable parameter's .grad against oracle autograd on the CPU.  Measured: value 5.6e-13,
    gradients 1.8e-12 relmax (C1); C4 <= 2.4e-15."""
    import types

    import api_builders as AB
    import helpers as Hh
    import mcpilco_b200.gpr_lib.Likelihood.Gaussian_likelihood as LK
    import mcpilco_b200.model_learning.Model_learning as ML
    R = types.SimpleNamespace(ML=ML)
    sc = W.real_shape(key, with_noise=False)
    ml = AB.build_model(R, sc, DEV, pretrain=False)
    crit = LK.Marginal_log_likelihood()
    X = Hh.T(sc["X"])
    for e, (gp, sp) in enumerate(zip(ml.gp_list, Hh.oracle_specs(sc))):
        loss = crit(gp(ml.gp_inputs), ml.gp_output_list[e])
        loss.backward()
        leaves = [sp["se"]["log_ls"].requires_grad_(True), sp["sigma_n_log"].requires_grad_(True)] + [m["log_par"].requires_grad_(True) for m in sp["mpk"]]
        ref = O.nlml(sp, X, Hh.T(sc["Y"][:, e:e + 1]))
        grads = torch.autograd.grad(ref.sum(), leaves)
        pre = "gp_list.0." if sp["mpk"] else ""
        want = {pre + "log_lengthscales_par": grads[0], pre + "sigma_n_log": grads[1]}
        want.update({"gp_list.1.gp_list.%d.Sigma_pos_par" % k: grads[2 + k] for k in range(len(sp["mpk"]))})
        got = {nm: p.grad for nm, p in gp.named_parameters() if p.requires_grad}
        assert set(got) == set(want)
        errs = {nm: relmax(got[nm].cpu().numpy().reshape(-1), want[nm].numpy().reshape(-1)) for nm in want}
        print("%s gp %d  nlml %.6e  value rel %.2e  worst grad %.2e" % (key, e, float(ref), abs(float(loss.detach()) / float(ref) - 1), max(errs.values())))
        assert abs(float(loss.detach()) - float(ref)) <= 1e-9 * abs(float(ref))
        assert max(errs.values()) <= 1e-6, errs


@pytest.mark.gpu
def test_sizes_reach_intended_kernels(gpu):
    """The sizes above were chosen from the dispatch thresholds of the precompute's products and of the NLML gradient kernel; this
    pins them to the kernels actually launched (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile

    def launched(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return {ev.name for ev in prof.events()}

    names = {}
    for N in (400, 1300, 2880, 3008, 4160):
        spec, X, y = cartpole_problem(N)
        Xg, yg = X.to(gpu), y.to(gpu)
        names[N] = launched(lambda: ops.gp_precompute(spec, Xg, yg))
    spec, X, y = well_problem(400, 24, "se_lin")
    names["nlml24"] = launched(lambda: ops.gp_nlml(spec, X.to(gpu), y.to(gpu)))
    if not any(names.values()):
        pytest.skip("the profiler recorded no CUDA activity")

    def has(key, pattern):
        return any(pattern in n for n in names[key])

    for N in (1300, 2880, 3008, 4160):
        assert has(N, "dgemm_tma_kernel<true>"), (N, sorted(names[N]))
    assert not has(400, "dgemm_tma_kernel"), sorted(names[400])
    assert has(1300, "dgemm_nt_kernel<64, 64, 2, 2>"), sorted(names[1300])
    assert has("nlml24", "nlml_grad_kernel<24>"), sorted(names["nlml24"])
