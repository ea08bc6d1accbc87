"""CPU: the shared library loads, exports every symbol include/mcpilco_b200.h declares, and the ctypes mirrors have the
library's struct layout.  No compute entry point is called (no GPU here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    from mcpilco_b200 import _build, _native
    _build.build()
    return _native


def test_header_symbols_exported(native):
    hdr = open(os.path.join(ROOT, "include", "mcpilco_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(mcpilco_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(native.SYMBOLS), declared ^ set(native.SYMBOLS)
    L = C.CDLL(native.LIB_PATH)
    for s in declared:
        assert hasattr(L, s), s


def test_abi_version_and_struct_layout(native):
    L = native.lib()  # raises on ABI or struct-size mismatch
    assert L.mcpilco_abi_version() == native.ABI_VERSION
    assert L.mcpilco_launch_count(0) == 0


def test_header_limits_match_binding(native):
    hdr = open(os.path.join(ROOT, "include", "mcpilco_b200.h")).read()
    for name, val in (("MCP_MAX_D", native.MAX_D), ("MCP_MAX_DS", native.MAX_DS), ("MCP_MAX_DU", native.MAX_DU),
                      ("MCP_MAX_E", native.MAX_E), ("MCP_MAX_DP", native.MAX_DP), ("MCP_MAX_POLY", native.MAX_POLY),
                      ("MCP_MAX_DEG", native.MAX_DEG), ("MCP_ABI_VERSION", native.ABI_VERSION),
                      ("MCP_OZAKI_EXP_NONFINITE", native.OZAKI_EXP_NONFINITE)):
        assert int(re.search(r"#define\s+%s\s+(\d+)" % name, hdr).group(1)) == val


def test_no_device_is_a_loud_error(native):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = native.lib()
    sm = C.c_int(0)
    assert L.mcpilco_device_info(C.byref(sm), None, None) == -2  # MCP_E_CUDA
    assert b"failed" in L.mcpilco_last_error()
    from mcpilco_b200 import _ops, _pack
    spec = _pack.spec_from_dict({"D": 2, "log_ls": [0.0, 0.0], "sigma_n": 0.1})
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _ops.gp_covariance(spec, torch.zeros(3, 2, dtype=torch.float64))


def test_spec_flattening_matches_oracle_closed_form():
    """_pack turns reference-style log-parameters into the closed form k(x,y) the kernels evaluate; check that closed form
    (evaluated here in numpy from the packed struct) against the oracle's reference-ordered computation."""
    import torch
    from mcpilco_b200 import _native as N, _pack as P
    from oracle import mcpilco_oracle as O
    rs = np.random.RandomState(0)
    D = 6
    log_ls = rs.randn(D)
    mpk = [np.exp(rs.randn(D + 1) - 3), np.exp(rs.randn(2 * D) - 3), np.exp(rs.randn(3 * D) - 3)]
    s = P.spec_from_dict({"D": D, "log_ls": log_ls, "lambda": 1.7, "mean": 0.3, "mpk": mpk, "sigma_n": 0.05, "sigma_n_num": 0.01})
    so = O.make_spec(D, log_ls=log_ls, log_lambda=np.log(1.7), mean=0.3, mpk_log_pars=[np.log(w) for w in mpk], sigma_n=0.05,
                     sigma_n_num=0.01)
    X1, X2 = rs.randn(5, D), rs.randn(7, D)

    def k_packed(x, y):
        v = 0.0
        if s.has_se:
            v += s.lambda_ * np.exp(-sum(((x[j] - y[j]) * s.inv_ls[j]) ** 2 for j in range(D)))
        for p in range(s.n_poly):
            pr = 1.0
            for f in range(N.MAX_DEG):
                pr *= sum(s.poly_w2[p][f][j] * x[j] * y[j] for j in range(D)) + s.poly_w2[p][f][N.MAX_D]
            v += pr
        return v
    K = np.array([[k_packed(a, b) for b in X2] for a in X1])
    Ko = O.gp_cov(so, torch.tensor(X1), torch.tensor(X2)).numpy()
    np.testing.assert_allclose(K, Ko, rtol=1e-12)
    assert abs(s.sigma_n2 - float(O.sigma_n2(so))) < 1e-16 and s.mean0 == 0.3 and list(s.poly_deg) == [1, 2, 3]


def test_struct_builders_validate():
    from mcpilco_b200 import _pack as P
    with pytest.raises(ValueError):
        P.new_gp_spec(0)
    with pytest.raises(ValueError):
        P.add_mpk(P.new_gp_spec(4), np.arange(4), 2, False, np.zeros(5))
    with pytest.raises(ValueError):
        P.model_struct("speed", 4, 1, 2, angle=[2], not_angle=[0, 1, 3], vel=[1], pos=[0, 2], T=0.05)
    m = P.model_struct("speed", 4, 1, 2, angle=[2], not_angle=[0, 1, 3], vel=[1, 3], pos=[0, 2], T=0.05)
    assert (m.D, m.n_na, m.n_a, m.kind, m.use_trig) == (6, 3, 1, 1, 1)
    ms = P.meas_struct([0, 2], [1, 3], [3e-3, 3e-3], 0.5, 1 / 30)
    assert abs(ms.b0 - 0.5) < 1e-15 and abs(ms.a1) < 1e-15 and ms.enabled == 1


def test_class_kernel_terms_match_flat_packing():
    """The class layer describes a kernel as differentiable torch terms (GP_prior._kernel_terms); the spec derived from them must be
    the one _pack builds from the flat dict (itself checked against the oracle above)."""
    import mcpilco_b200.gpr_lib.GP_prior.GP_prior as GP
    import mcpilco_b200.gpr_lib.GP_prior.Sparse_GP as SP
    import mcpilco_b200.gpr_lib.GP_prior.Stationary_GP as SGP
    from mcpilco_b200 import _pack as P
    rs = np.random.RandomState(1)
    D = 7
    act_se, act_mpk = np.array([0, 2, 3, 5]), np.array([1, 2, 6])
    log_ls = rs.randn(4)
    mpk = [np.exp(rs.randn(4) - 3), np.exp(rs.randn(6) - 3)]
    rbf = SGP.RBF(act_se, lengthscales_init=np.exp(log_ls), lambda_init=np.array([0.7]), sigma_n_init=np.array([0.2]), mean_init=np.array([-0.4]),
                  sigma_n_num=1e-3)
    vol = SP.get_Volterra_MPK_GP(act_mpk, 2, Sigma_pos_par_init_list=mpk, flg_train_Sigma_pos_par_list=[True, True])
    s = GP.Sum_Independent_GP(rbf, vol).gp_spec(D)
    ref = P.new_gp_spec(D)
    P.add_se(ref, act_se, log_ls, np.log(0.7), -0.4)
    P.add_mpk(ref, act_mpk, 1, True, np.log(mpk[0]))
    P.add_mpk(ref, act_mpk, 2, False, np.log(mpk[1]))
    assert (s.has_se, s.n_poly, list(s.poly_deg)) == (1, 2, [1, 2, 0]) and abs(s.lambda_ - 0.7) < 1e-15 and s.mean0 == -0.4
    np.testing.assert_allclose(np.array(s.inv_ls), np.array(ref.inv_ls), rtol=1e-14)
    np.testing.assert_allclose(np.ctypeslib.as_array(s.poly_w2), np.ctypeslib.as_array(ref.poly_w2), rtol=1e-13)
    assert abs(s.sigma_n2 - (0.2 ** 2 + 1e-6)) < 1e-15
    # a scalar (non-ARD) lengthscale broadcasts over the active dimensions
    iso = SGP.RBF(np.arange(3), lengthscales_init=np.array([2.0]), sigma_n_init=np.array([0.1])).gp_spec(3)
    assert list(iso.inv_ls)[:3] == [0.5, 0.5, 0.5]


def test_argument_errors_are_reported_before_any_cuda_work(native):
    """Entry points validate their arguments first: bad shapes / null pointers return MCP_E_ARG with a message, on a box with or
    without a GPU (nothing is launched)."""
    from mcpilco_b200 import _pack as P
    L = native.lib()
    spec = P.spec_from_dict({"D": 3, "log_ls": [0.0, 0.0, 0.0], "sigma_n": 0.1})
    E_ARG = -1
    assert L.mcpilco_gp_covariance(None, None, 4, None, 4, 0, None, 4, None) == E_ARG and b"null gp spec" in L.mcpilco_last_error()
    bad = P.spec_from_dict({"D": 3, "log_ls": [0.0, 0.0, 0.0], "sigma_n": 0.1}); bad.D = 99
    assert L.mcpilco_gp_covariance(C.byref(bad), None, 4, None, 4, 0, None, 4, None) == E_ARG and b"gp input dim 99" in L.mcpilco_last_error()
    empty = P.new_gp_spec(3)
    assert L.mcpilco_gp_diag_covariance(C.byref(empty), None, 4, None, None) == E_ARG and b"empty kernel" in L.mcpilco_last_error()
    assert L.mcpilco_gp_precompute(C.byref(spec), None, None, 0, None, None, 0, None, None, None, 0, None) == E_ARG
    assert L.mcpilco_gp_predict(None, 0, None, 5, None, None, None, None, None, 0, None) == E_ARG and b"bad E" in L.mcpilco_last_error()
    assert L.mcpilco_gp_nlml(C.byref(spec), None, None, 5, None, None, 0, None) == E_ARG
    assert L.mcpilco_gp_sod_select(C.byref(spec), None, 5, None, 0.1, None, None, None, 0, None) == E_ARG
    assert L.mcpilco_rollout_fwd(None, None) == E_ARG and b"null rollout descriptor" in L.mcpilco_last_error()
    r = native.Rollout()
    r.M, r.H = 0, 5
    assert L.mcpilco_rollout_fwd(C.byref(r), None) == E_ARG and b"M=0" in L.mcpilco_last_error()
    r.M = 4
    r.model.Ds, r.model.Du, r.model.E, r.model.D = 4, 1, 2, 7   # feature map would give 5
    assert L.mcpilco_rollout_fwd(C.byref(r), None) == E_ARG and b"does not match the feature map" in L.mcpilco_last_error()
    assert L.mcpilco_policy_forward(None, 3, 0, None, 0.0, None, 0, 0, None, None) == E_ARG
    assert L.mcpilco_init_particles(2, None, None, 1, 4, 4, 0, 0, None, None, None) == E_ARG
    assert L.mcpilco_ozaki_prepare(None, 4, 4, 8, None, None, None) == E_ARG
    # workspace queries are pure host arithmetic
    assert L.mcpilco_gp_precompute_workspace_bytes(300) > 2 * 320 * 320 * 8
    assert L.mcpilco_rollout_workspace_bytes(400, 60, 2, 6, 300, 200, 5, 1) > 0 and L.mcpilco_gp_nlml_grad_size() == 4 + 32 + 9 * 33
    assert L.mcpilco_ozaki_plane_bytes(8192, 8) == 8192 * 8 * 8192 and L.mcpilco_ozaki_plane_bytes(16384, 8) == 16384 * 2 * 8 * 8192


def test_torch_custom_ops_registered_and_shape_checked():
    """torch.ops.mcpilco.* exist, infer shapes on meta/fake tensors, and refuse CPU tensors (no CPU implementation)."""
    import torch
    from torch._subclasses.fake_tensor import FakeTensorMode
    from mcpilco_b200 import _pack as P
    from mcpilco_b200 import torch_ops as TO
    spec = P.spec_from_dict({"D": 3, "log_ls": [0.0, 0.1, 0.2], "sigma_n": 0.1, "mpk": [[[1.0, 2.0, 3.0, 0.5]]]})
    t = TO.spec_tensor(spec)
    back = TO._spec(t)
    assert bytes(back) == bytes(spec)
    for name in ("gp_covariance", "gp_diag_covariance", "gp_precompute", "gp_predict", "gp_predict_jac", "gp_nlml"):
        assert hasattr(torch.ops.mcpilco, name)
    with FakeTensorMode(allow_non_fake_inputs=True):
        X, Xs = torch.empty(10, 3, dtype=torch.float64), torch.empty(7, 3, dtype=torch.float64)
        y = torch.empty(10, 1, dtype=torch.float64)
        assert torch.ops.mcpilco.gp_covariance(t, X, Xs, False).shape == (10, 7)
        a, Ki = torch.ops.mcpilco.gp_precompute(t, X, y)
        assert a.shape == (10, 1) and Ki.shape == (10, 10)
        m, v, jm, jv = torch.ops.mcpilco.gp_predict_jac(t, X, a, Ki, Xs, 1.0)
        assert m.shape == (7, 1) and jv.shape == (7, 3)
        assert torch.ops.mcpilco.gp_nlml(t, X, y).numel() == 4 + 32 + 3 * 3 * 33
    with pytest.raises(NotImplementedError):
        torch.ops.mcpilco.gp_covariance(t, torch.zeros(4, 3, dtype=torch.float64), None, False)
    with pytest.raises(RuntimeError):
        TO._spec(torch.zeros(5, dtype=torch.uint8))
