"""The two small-shape rollout paths at every template instance and shape edge, against the CPU oracle.

The reference's real configurations (C1-C3, the first trial) run on one of two paths that the large per-step kernels never touch:
the whole-horizon cluster kernel `persist_rollout_kernel<DT, NP, JAC>` (csrc/mcp_persist.cu) and the fused two-launch step
`small_step_kernel<DT, NP, JAC>` + `small_gemm_kernel` (csrc/mcp_small.cu).  Both are templates over fixed-size register and shared
memory arrays with padded tiles and hand-written copy tails.  Each case below is a seeded synthetic scenario (tests/scenarios.py
format) run on every path it is eligible for:

  persistent   MCPILCO_PERSIST=1       the cluster kernel wherever it is eligible, whatever the default heuristic says
  fused-small  MCPILCO_NO_PERSIST=1    the fused two-launch step
  per-step     MCPILCO_NO_SMALL_PATH=1 the per-step kernels of the large shapes
  default      no switch               the default dispatch (only where its choice is documented: the flips below)

The grid: every (DT, NP) instance of both templates with and without the Jacobian checkpoints (JAC = need_grad); odd and even
training-set sizes N = 1 ... 301 with E = 1, 2, 4 outputs; N at the cluster kernel's shared-memory limit and one above it; control
inputs Du = 1 ... 4 and GP input widths D = 2 ... 8; particle counts around the 27-particle cluster batch; horizons H = 1 and 2;
the default-dispatch flips; and outputs with training sets of different sizes (per-output subset-of-data models).

Checks per case:
  * formula level: the oracle's fp64 alpha and K^-1 go into the CUDA rollout, so precompute conditioning is out of the comparison;
    states, inputs, cost, std_cost (M >= 2) and the log_ls / centers / W / bias gradients against oracle autograd;
  * cross-path: every path agrees with the others on the same inputs;
  * no-grad: the need_grad=False rollout (JAC = false instance) matches the need_grad=True one;
  * own precompute (per-output-size cases): the CUDA factors end to end, at the north-star tolerances;
  * the launched kernel names (torch.profiler) name the intended path and <DT, NP, JAC> instance, so a dispatch change cannot move a
    case to another path unnoticed; a final test asserts that every instance of both templates was reached.  The profiled runs of
    all cases happen in one child process: late in a long pytest process the profiler was seen to drop kernel records of sessions
    that contain the cluster kernel (the library's own launch counter showed the cluster path was taken), and a fresh process
    makes the check independent of what ran before.

Bounds are about 10x the largest error measured on a B200 (1000 W power limit) over the whole grid:
  formula level   states / inputs 1.7e-9, cost 3.6e-10, std_cost 7.6e-10, gradients 5.6e-9   (max |a - b| / max |b|)
  cross-path      states / inputs 1.7e-9, cost 6.0e-10, gradients 8.5e-9
  no-grad         states / inputs 7.1e-11, cost 1.1e-11
  own precompute  states 9.2e-10, cost 1.5e-10, std_cost 1.6e-9, gradients 3.0e-9; the bounds are the north star's (1e-5, 1e-4)
  class level     states 1.2e-12, gradients 1.8e-13 (north-star bounds)
The largest errors come from the worst-conditioned cases (N = 299 points in two dimensions, N = 2048 / 2049): they are the
oracle's and the kernels' rounding amplified by the cancellation in the posterior variance, so the paths differ from one another
by as much as from the oracle.  The single-line kernel defects this file was checked against (a dropped odd-N copy, a wrong
output's N, a dropped Volterra offset, one control input written instead of Du) moved results by 1e-2 or more, or to NaN."""
import math

import numpy as np
import pytest
import torch

import helpers as Hh
from oracle import mcpilco_oracle as O

pytestmark = pytest.mark.gpu

# formula level (oracle factors in), cross-path, no-grad; see the module docstring for the measured maxima
TOL_TRAJ, TOL_COST, TOL_STD, TOL_GRAD = 2e-8, 4e-9, 8e-9, 6e-8
TOL_XPATH_TRAJ, TOL_XPATH_COST, TOL_XPATH_GRAD = 2e-8, 6e-9, 9e-8
TOL_NOGRAD_TRAJ, TOL_NOGRAD_COST = 7e-10, 1e-10
REL_VAL, REL_GRAD = 1e-5, 1e-4   # north star (own precompute)

# Largest training-set size whose K^-1 slices fit the cluster kernel's 227 KB of shared memory, per output count E: from
# pk_geom(N, E) in csrc/mcp_persist.cu (N is rounded up to 16, so N + 1 is the first size that does not fit).  Hard-coded so that a
# change of the kernel's geometry fails these tests instead of silently moving the limit cases off the limit.
PK_SMEM_N_LIMIT = {1: 304, 2: 304, 3: 288, 4: 272}

ENV_VARS = ("MCPILCO_NO_SMALL_PATH", "MCPILCO_NO_BATCHED_STEP", "MCPILCO_NO_PDL", "MCPILCO_NO_PERSIST", "MCPILCO_PERSIST")
PATHS = {"persistent": {"MCPILCO_PERSIST": "1"}, "fused-small": {"MCPILCO_NO_PERSIST": "1"}, "per-step": {"MCPILCO_NO_SMALL_PATH": "1"},
         "default": {}}

_oracle_cache = {}
MEASURED = {}      # metric -> largest error seen in this session
REACHED = set()    # kernel instances seen in the profiler
PROFILED = []      # False once the profiler recorded no CUDA activity


@pytest.fixture(scope="module")
def nh():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import native_helpers
    return native_helpers


# ---------------------------------------------------------------------------------------------------------------------
# seeded synthetic scenarios
# ---------------------------------------------------------------------------------------------------------------------
def _noise(sc, rs):
    M, H, nb = sc["M"], sc["H"], sc["policy"]["nb"]
    sc["eps0"] = rs.randn(M, sc["Ds"])
    sc["eps"] = rs.randn(H - 1, M, sc["E"])
    sc["masks"] = (rs.rand(H, M, nb) >= sc["p_dropout"]).astype(np.float64)
    if "pms" in sc:
        sc["meas_eps"] = rs.randn(H - 1, M, len(sc["pms"]["pos_idx"]))
    return sc


def _gp_pars(rs, D, n_poly, e):
    """SE + n_poly Volterra terms (spec_from_dict: D + 1 values for degree 1, which has the offset, 2 D for degree 2)."""
    mpk = []
    if n_poly >= 1:
        mpk.append(0.2 * np.exp(0.1 * rs.randn(D + 1)))
    if n_poly >= 2:
        mpk.append(0.2 * np.exp(0.1 * rs.randn(2 * D)))
    return {"log_ls": math.log(1.2) + 0.1 * rs.randn(D), "lambda": 0.8 + 0.4 * rs.rand(), "sigma_n": 0.05 + 0.05 * rs.rand(),
            "mean": 0.01 * (e + 1), "mpk": mpk}


def _policy(rs, kind, nb, Ds, Du, H):
    if kind == "plain":   # bias and input scale, no squashing
        return {"kind": "plain", "nb": nb, "centers": rs.uniform(-1, 1, (nb, Ds)), "lengthscales": 1.0 + rs.rand(Ds),
                "weight": rs.rand(Du, nb) - 0.5, "u_max": None, "bias": 0.05 * rs.randn(Du), "scale": 0.5 + rs.rand(Ds)}
    if kind == "angles":  # state 0 is an angle: features [x_1.., cos x_0, sin x_0], squashed
        ang = np.pi * 2 * (rs.rand(nb, 1) - 0.5)
        return {"kind": "angles", "nb": nb, "centers": np.concatenate([rs.uniform(-1, 1, (nb, Ds - 1)), np.cos(ang), np.sin(ang)], 1),
                "lengthscales": 1.0 + 0.3 * rs.rand(Ds + 1), "weight": 2.0 * (rs.rand(Du, nb) - 0.5), "u_max": 2.0,
                "angle": np.array([0]), "non_angle": np.arange(1, Ds), "bias": None, "scale": None}
    tt = np.linspace(0, 1, H)[:, None]   # "target": features [x, target_t - x], squashed per input
    traj = 0.2 * np.sin(2 * tt + 0.5 * np.arange(Ds)[None])
    return {"kind": "target", "nb": nb, "centers": 0.5 * rs.uniform(-1, 1, (nb, 2 * Ds)), "lengthscales": 1.5 * np.ones(2 * Ds),
            "weight": 2.0 * (rs.rand(Du, nb) - 0.5), "u_max": [1.0] * Du, "target_traj": traj, "bias": None, "scale": None}


def synthetic(E=2, Du=1, n_poly=0, policy="plain", N=47, M=9, H=3, nb=12, seed=0):
    """Delta-state model with Ds = E states, Du inputs and gp inputs [x, u] (D = E + Du), well conditioned: inputs of order 1,
    sigma_n in [0.05, 0.1].  N an int (one training set) or one size per output: output e then trains on its own row subset X_e."""
    rs = np.random.RandomState(5000 + seed)
    Ds, D = E, E + Du
    Ns = (int(N),) * E if np.isscalar(N) else tuple(int(n) for n in N)
    assert len(Ns) == E
    Nall = max(Ns)
    X = rs.uniform(-1, 1, (Nall, D))
    A, B = rs.randn(D, E) / math.sqrt(D), rs.randn(D, E) / math.sqrt(D)
    Y = 0.05 * (np.sin(X @ A + 0.3) + 0.5 * np.cos(2 * X @ B)) + 0.01 * rs.randn(Nall, E)
    rows = [np.sort(rs.choice(Nall, n, replace=False)) for n in Ns]
    sc = dict(name="synthetic", D=D, Ds=Ds, Du=Du, E=E, N=Nall, M=M, H=H, X=X, Y=Y, rows=rows,
              gps=[_gp_pars(rs, D, n_poly, e) for e in range(E)],
              model={"kind": "delta", "use_trig": False, "angle": [], "not_angle": list(range(Ds)), "vel": [], "pos": [], "T": 0.0},
              policy=_policy(rs, policy, nb, Ds, Du, H), p_dropout=0.1,
              cost={"kind": "sat_target", "target": 0.1 * np.ones((1, min(Ds, 2))), "ls": np.ones(min(Ds, 2)),
                    "active": list(range(min(Ds, 2)))},
              x0_mean=0.1 * rs.randn(Ds), x0_var=1e-3 * np.ones(Ds))
    return _noise(sc, rs)


def cartpole(key="c1", n_poly=2, N=64, M=27, H=4, nb=20, seed=0):
    """Cart-pole speed model (E = 2, D = 6) of the real-shape tests; "c3" adds the 4PMS measurement model (SE-only), "c1" has the
    SE + Volterra kernels (n_poly = 1 keeps the degree-1 term only)."""
    from mcpilco_b200 import workloads as W
    sc = W.real_shape(key, seed=seed, N=N, M=M, H=H, nb=nb)
    for g in sc["gps"]:
        g["mpk"] = list(g["mpk"][:n_poly])
    sc["rows"] = [np.arange(N)] * 2
    return sc


def build(spec):
    kw = dict(spec)
    return cartpole(**kw["cartpole"]) if "cartpole" in kw else synthetic(**kw)


def dims(spec):
    """(D, n_poly) of a case without building its data."""
    if "cartpole" in spec:
        return 6, spec["cartpole"].get("n_poly", 2)
    return spec.get("E", 2) + spec.get("Du", 1), spec.get("n_poly", 0)


# ---------------------------------------------------------------------------------------------------------------------
# the case grid: (path, kernel family expected there); "persist" = the cluster kernel, "small" = the fused step, "step" = neither
# ---------------------------------------------------------------------------------------------------------------------
ALL3 = (("persistent", "persist"), ("fused-small", "small"), ("per-step", "step"))
NO_PK = (("persistent", "small"), ("fused-small", "small"), ("per-step", "step"))   # the cluster kernel refuses the case
BOTH = (True, False)
CASES = {}


def _case(cid, paths, grads=(True,), own=False, **spec):
    CASES[cid] = dict(spec=spec, paths=paths, grads=grads, own=own)


# every (DT, NP) instance of both templates, with and without the Jacobian checkpoints
_case("inst-dt4-np0", ALL3, BOTH, E=2, Du=1, n_poly=0, policy="plain", N=47, M=28, H=4)
_case("inst-dt4-np1", ALL3, BOTH, E=1, Du=3, n_poly=1, policy="angles", N=129, M=27, H=3)
_case("inst-dt4-np2", ALL3, BOTH, E=3, Du=1, n_poly=2, policy="target", N=17, M=26, H=3)
_case("inst-dt6-np0-4pms", ALL3, BOTH, cartpole=dict(key="c3", n_poly=0, N=61, M=27, H=4))
_case("inst-dt6-np1", ALL3, BOTH, E=4, Du=2, n_poly=1, policy="plain", N=15, M=12, H=3)
_case("inst-dt6-np2", ALL3, BOTH, E=2, Du=3, n_poly=2, policy="angles", N=301, M=9, H=3)
_case("inst-dt6-np2-cartpole", ALL3, BOTH, cartpole=dict(key="c1", n_poly=2, N=64, M=27, H=4))
_case("inst-dt6-np1-cartpole", ALL3, BOTH, cartpole=dict(key="c1", n_poly=1, N=48, M=9, H=3))
_case("inst-dt8-np0", NO_PK, BOTH, E=4, Du=3, n_poly=0, policy="target", N=47, M=9, H=3)
_case("inst-dt8-np1", NO_PK, BOTH, E=4, Du=4, n_poly=1, policy="plain", N=129, M=9, H=3)
# control inputs Du = 1 ... 4 and gp input widths D = 2, 3, 5, 7 (padded features of the wider instance)
_case("dims-D2-Du1", ALL3, E=1, Du=1, n_poly=2, policy="target", N=47)
_case("dims-D3-Du2", ALL3, E=1, Du=2, n_poly=0, policy="plain", N=33)
_case("dims-D5-Du4", ALL3, E=1, Du=4, n_poly=1, policy="plain", N=47)
_case("dims-D6-Du4", ALL3, E=2, Du=4, n_poly=0, policy="angles", N=31)
_case("dims-D5-Du3", ALL3, E=2, Du=3, n_poly=1, policy="target", N=40)
_case("dims-D7-Du4", NO_PK, E=3, Du=4, n_poly=1, policy="angles", N=47)
# odd and even training-set sizes: the cluster kernel's odd-last-element copy, the small GEMM's 8-byte cp.async tail, N < one tile
for _i, _n in enumerate((1, 15, 17, 47, 129, 299, 301)):
    for _E, _Du in ((1, 1), (2, 2), (4, 1)):
        _paths = ALL3 if _n <= PK_SMEM_N_LIMIT[_E] else NO_PK
        _case("N%d-E%d" % (_n, _E), _paths, E=_E, Du=_Du, n_poly=(_i + _E) % 3, policy=("plain", "angles", "target")[(_i + _E) % 3],
              N=_n, M=9, H=3, seed=_i)
# the cluster kernel's shared-memory limit and one above it (forced: it must then not be taken)
for _E, _n in PK_SMEM_N_LIMIT.items():
    _case("smem-limit-E%d-N%d" % (_E, _n), (("persistent", "persist"), ("fused-small", "small")), E=_E, Du=1, n_poly=1, N=_n, M=9, H=2)
    _case("smem-over-E%d-N%d" % (_E, _n + 1), (("persistent", "small"), ("fused-small", "small")), E=_E, Du=1, n_poly=1, N=_n + 1, M=9, H=2)
# particle counts around one 27-particle cluster batch
for _m in (1, 26, 27, 28):
    _case("M%d" % _m, (("persistent", "persist"), ("fused-small", "small")), E=2, Du=2, n_poly=1, policy="angles", N=47, M=_m, H=3)
# horizons: 2 is the cluster kernel's smallest; it refuses 1
_case("H2", ALL3, E=2, Du=1, n_poly=2, policy="plain", N=47, M=9, H=2)
_case("H1-M1", NO_PK, BOTH, E=2, Du=1, n_poly=1, policy="plain", N=47, M=1, H=1)
_case("H1-M9", NO_PK, BOTH, E=2, Du=1, n_poly=0, policy="angles", N=47, M=9, H=1)
# default-dispatch flips (no switch set): SE-only N <= 240 on the cluster kernel; one pass of 15 co-resident clusters x 27 = 405
# particles at N = 300 (DESIGN.md section 6: 15 clusters once a CTA needs more than 113 KB); the small path's N <= 2048
_case("flip-se-N240", (("default", "persist"),), E=2, Du=2, n_poly=0, policy="plain", N=240, M=27, H=2)
_case("flip-se-N241", (("default", "small"),), E=2, Du=2, n_poly=0, policy="plain", N=241, M=27, H=2)
_case("flip-M405", (("default", "persist"),), cartpole=dict(key="c1", n_poly=2, N=300, M=405, H=2))
_case("flip-M406", (("default", "small"),), cartpole=dict(key="c1", n_poly=2, N=300, M=406, H=2))
_case("flip-N2048", (("default", "small"),), E=1, Du=2, n_poly=1, policy="plain", N=2048, M=4, H=2)
_case("flip-N2049", (("default", "step"),), E=1, Du=2, n_poly=1, policy="plain", N=2049, M=4, H=2)
# outputs with training sets of different sizes (per-output subset of data): the cluster kernel must refuse them
_case("ragged-300-257", NO_PK, BOTH, own=True, E=2, Du=1, n_poly=1, policy="plain", N=(300, 257), M=9, H=3)
_case("ragged-61-200-129", NO_PK, BOTH, own=True, E=3, Du=2, n_poly=2, policy="angles", N=(61, 200, 129), M=9, H=3)
_case("ragged-17-301-64-255", NO_PK, BOTH, own=True, E=4, Du=1, n_poly=0, policy="target", N=(17, 301, 64, 255), M=9, H=3)
_case("ragged-2048-1500", NO_PK, own=True, E=2, Du=2, n_poly=1, policy="plain", N=(2048, 1500), M=4, H=3)


def instance(family, D, n_poly, jac):
    if family == "persist":
        return "persist_rollout_kernel<%d, %d, %s>" % (4 if D <= 4 else 6, n_poly, "true" if jac else "false")
    return "small_step_kernel<%d, %d, %s>" % (4 if D <= 4 else (6 if D <= 6 else 8), n_poly, "true" if jac else "false")


ALL_INSTANCES = ({instance("persist", D, p, j) for D in (4, 6) for p in range(3) for j in BOTH} |
                 {instance("small", D, p, j) for D in (4, 6, 8) for p in range(3) for j in BOTH if not (D == 8 and p == 2)})


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def relmax(a, b):
    a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
    b = b.detach().cpu().numpy() if hasattr(b, "detach") else np.asarray(b)
    return float(np.abs(a.reshape(b.shape) - b).max() / max(np.abs(b).max(), 1e-300))


def note(metric, err):
    MEASURED[metric] = max(MEASURED.get(metric, 0.0), err)
    return err


def set_path(monkeypatch, path):
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)


def oracle_factors(sc):
    """Oracle fp64 factors per output: (spec, X_e, alpha_e, K^-1_e)."""
    torch.set_num_threads(max(1, min(16, torch.get_num_threads())))
    gps = []
    for e, sp in enumerate(Hh.oracle_specs(sc)):
        r = sc["rows"][e]
        Xe = Hh.T(sc["X"][r])
        alpha, _, Kinv = O.gp_fit(sp, Xe, Hh.T(sc["Y"][r, e:e + 1]))
        gps.append((sp, Xe, alpha, Kinv))
    return gps


def oracle_of(key, sc):
    """Oracle fp64 factors per output and the oracle rollout on them (cached per scenario)."""
    if key not in _oracle_cache:
        gps = oracle_factors(sc)
        _oracle_cache[key] = (gps, Hh.oracle_rollout(sc, gps=gps, requires_grad=sc["H"] > 1))
    return _oracle_cache[key]


def native_gps(nh, sc, ogps=None):
    """FittedGp per output on its own rows: the oracle's factors when given (formula level), else the CUDA precompute."""
    from mcpilco_b200 import _ops as ops
    gps = []
    for e, sp in enumerate(nh.native_specs(sc)):
        r = sc["rows"][e]
        Xe = nh.G(sc["X"][r])
        if ogps is not None:
            gps.append(ops.FittedGp(sp, Xe, nh.G(ogps[e][2].numpy()), nh.G(ogps[e][3].numpy())))
        else:
            alpha, Kinv, Linv = ops.gp_precompute(sp, Xe, nh.G(sc["Y"][r, e:e + 1]), want_Linv=True)
            gps.append(ops.FittedGp(sp, Xe, alpha, Kinv, Linv=Linv))
    return gps


def launched(fn):
    """Names of the CUDA kernels fn launched (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {ev.name for ev in prof.events()}


def run(nh, sc, gps, need_grad, profile=False):
    plan, _ = nh.native_plan(sc, gps, need_grad=need_grad)
    x0 = nh.x0_of(sc)
    names = launched(lambda: plan.forward(x0)) if profile else (plan.forward(x0), None)[1]
    out = {"states": plan.states.clone(), "inputs": plan.inputs.clone(), "cost": plan.cost_out[:2 if sc["M"] >= 2 else 1].clone()}
    if need_grad:
        gr = plan.backward(grad_cost=1.0)
        torch.cuda.synchronize()
        out.update({"g_" + k: v.clone() for k, v in gr.items() if v is not None})
    torch.cuda.synchronize()
    return out, names


def check_kernels(names, family, D, n_poly, jac, tag):
    if not names:
        PROFILED.append(False)
        return
    PROFILED.append(True)
    pk = sorted(n for n in names if "persist_rollout_kernel" in n)
    ss = sorted(n for n in names if "small_step_kernel" in n)
    if family == "persist":
        want = instance("persist", D, n_poly, jac)
        assert pk and all(want in n for n in pk) and not ss, (tag, want, pk, ss)
    elif family == "small":
        want = instance("small", D, n_poly, jac)
        assert ss and all(want in n for n in ss) and not pk, (tag, want, pk, ss)
    else:
        want = None
        assert not pk and not ss, (tag, pk, ss)
    if want is not None:
        REACHED.add(want)


def compare_oracle(out, ref, sc, need_grad, tag, tols):
    t_traj, t_cost, t_std, t_grad, kind = tols
    errs = {"states": relmax(out["states"], ref["states"]), "inputs": relmax(out["inputs"], ref["inputs"]),
            "cost": abs(float(out["cost"][0]) - float(ref["cost"])) / abs(float(ref["cost"]))}
    if sc["M"] >= 2:
        errs["std_cost"] = abs(float(out["cost"][1]) - float(ref["std_cost"])) / abs(float(ref["std_cost"]))
    if need_grad:
        for k in ("log_ls", "centers", "W", "bias"):
            if "g_" + k in ref:
                errs["g_" + k] = relmax(out["g_" + k], ref["g_" + k])
            elif "g_" + k in out:    # H = 1: the cost does not depend on the policy
                errs["g_" + k] = float(out["g_" + k].abs().max())
    for k, v in errs.items():
        note("%s/%s" % (kind, "grad" if k.startswith("g_") else k), v)
    print(tag, kind, {k: "%.1e" % v for k, v in errs.items()})
    assert not torch.isnan(out["states"]).any(), tag
    assert errs["states"] <= t_traj and errs["inputs"] <= t_traj and errs["cost"] <= t_cost, (tag, errs)
    assert errs.get("std_cost", 0.0) <= t_std, (tag, errs)
    assert max([v for k, v in errs.items() if k.startswith("g_")] + [0.0]) <= t_grad, (tag, errs)


def compare_runs(a, b, tag, kind, t_traj, t_cost, t_grad):
    errs = {k: relmax(a[k], b[k]) for k in a if k in b}
    for k, v in errs.items():
        note("%s/%s" % (kind, "grad" if k.startswith("g_") else ("cost" if k == "cost" else "traj")), v)
    assert errs["states"] <= t_traj and errs["inputs"] <= t_traj and errs["cost"] <= t_cost, (tag, kind, errs)
    assert max([v for k, v in errs.items() if k.startswith("g_")] + [0.0]) <= t_grad, (tag, kind, errs)


# ---------------------------------------------------------------------------------------------------------------------
# the grid
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cid", list(CASES))
def test_small_path_case_vs_oracle(nh, monkeypatch, cid):
    c = CASES[cid]
    sc = build(c["spec"])
    D, n_poly = sc["D"], len(sc["gps"][0]["mpk"])
    ogps, ref = oracle_of(cid, sc)
    runs = {}
    for path, family in c["paths"]:
        set_path(monkeypatch, path)
        for need_grad in c["grads"]:
            tag = "%s/%s/%s" % (cid, path, "grad" if need_grad else "nograd")
            out, _ = run(nh, sc, native_gps(nh, sc, ogps), need_grad)
            compare_oracle(out, ref, sc, need_grad, tag, (TOL_TRAJ, TOL_COST, TOL_STD, TOL_GRAD, "formula"))
            runs[(path, need_grad)] = out
        if False in c["grads"] and True in c["grads"]:
            g, ng = runs[(path, True)], runs[(path, False)]
            compare_runs({k: ng[k] for k in ("states", "inputs", "cost")}, g, cid + "/" + path, "nograd", TOL_NOGRAD_TRAJ, TOL_NOGRAD_COST, 0.0)
        if c["own"]:
            out, _ = run(nh, sc, native_gps(nh, sc), True)
            compare_oracle(out, ref, sc, True, "%s/%s/own" % (cid, path), (REL_VAL, REL_VAL, 1e-4, REL_GRAD, "own"))
    keys = sorted(runs)
    for i, ka in enumerate(keys):
        for kb in keys[i + 1:]:
            if ka[1] == kb[1] and ka[0] != kb[0]:
                compare_runs(runs[ka], runs[kb], "%s %s~%s" % (cid, ka[0], kb[0]), "xpath", TOL_XPATH_TRAJ, TOL_XPATH_COST, TOL_XPATH_GRAD)


def test_sod_model_per_output_sizes_vs_oracle(nh):
    """Class level: a subset-of-data model (approximation_mode "SOD") whose outputs keep subsets of different sizes (per-output
    thresholds; about 170 and 50 of the 200 cart-pole points), through apply_policy with the 4PMS measurement model, the fused cost
    and cost.backward(), against the oracle fitted on each output's SOD_indices subset.  Own precompute: north-star tolerances."""
    import types
    import api_builders as AB
    import mcpilco_b200.model_learning.Model_learning as ML
    import mcpilco_b200.policy_learning.Cost_function as CF
    import mcpilco_b200.policy_learning.MC_PILCO as MCP
    import mcpilco_b200.policy_learning.Policy as PO
    from mcpilco_b200 import workloads as W
    R = types.SimpleNamespace(ML=ML, CF=CF, MCP=MCP, PO=PO)
    dev = torch.device("cuda:0")
    sc = W.real_shape("c3", N=200, M=27, H=5)
    ml = AB.build_model(R, sc, dev, approximation={"SOD_threshold_mode": "absolute", "SOD_threshold": [0.15, 0.5], "flg_SOD_permutation": False})
    idx = [np.array([int(i) for i in ml.SOD_indices[e]]) for e in range(sc["E"])]
    assert len(idx[0]) != len(idx[1]) and max(len(i) for i in idx) < sc["N"], [len(i) for i in idx]
    X = Hh.T(sc["X"])
    ogps = []
    for e, sp in enumerate(Hh.oracle_specs(sc)):
        alpha, _, Kinv = O.gp_fit(sp, X[idx[e]], Hh.T(sc["Y"][idx[e], e:e + 1]))
        ogps.append((sp, X[idx[e]], alpha, Kinv))
    ref = Hh.oracle_rollout(sc, gps=ogps)
    obj = AB.build_pilco(R, sc, ml, dev)
    T = AB.tensor_factory(dev)
    noise = dict(eps0=T(sc["eps0"]), eps=T(sc["eps"]), masks=T(sc["masks"]), meas_eps=T(sc["meas_eps"]))
    states, inputs = obj.apply_policy(**AB.apply_kwargs(sc, dev), _noise=noise)
    cost, std_cost = obj.cost_function(states, inputs, 0)
    cost.backward()
    pol = obj.control_policy
    errs = {"states": relmax(states, ref["states"]), "inputs": relmax(inputs, ref["inputs"]),
            "cost": abs(float(cost.detach()) / float(ref["cost"]) - 1), "std_cost": abs(float(std_cost) / float(ref["std_cost"]) - 1),
            "g_log_ls": relmax(pol.log_lengthscales.grad, ref["g_log_ls"]), "g_centers": relmax(pol.centers.grad, ref["g_centers"]),
            "g_W": relmax(pol.f_linear.weight.grad, ref["g_W"])}
    for k, v in errs.items():
        note("sod/%s" % ("grad" if k.startswith("g_") else k), v)
    print("sod sizes", [len(i) for i in idx], {k: "%.1e" % v for k, v in errs.items()})
    assert errs["states"] < REL_VAL and errs["inputs"] < REL_VAL and errs["cost"] < REL_VAL and errs["std_cost"] < 1e-4, errs
    assert max(errs["g_log_ls"], errs["g_centers"], errs["g_W"]) < REL_GRAD, errs


# every case and path of the grid, profiled in a fresh process (see the module docstring); prints {"cid|path|need_grad": [names]}
_PROFILE_SCRIPT = r"""
import json, os, sys
sys.path[:0] = SYS_PATH
import native_helpers as nh
import MODULE as T
out = {}
for cid, c in T.CASES.items():
    sc = T.build(c["spec"])
    gps = T.native_gps(nh, sc, T.oracle_factors(sc))
    for path, _ in c["paths"]:
        for v in T.ENV_VARS:
            os.environ.pop(v, None)
        os.environ.update(T.PATHS[path])
        for need_grad in c["grads"]:
            _, names = T.run(nh, sc, gps, need_grad, profile=True)
            out["%s|%s|%d" % (cid, path, need_grad)] = sorted(names)
print(json.dumps(out))
"""


def test_every_instance_is_reached():
    """Every case launches the intended path and <DT, NP, JAC> instance (the same inputs as the case's oracle comparison, profiled
    in a child process), every cluster-kernel instance (12) and small-step instance (16) is the expected kernel of some case, and
    each of them was seen in the profiler."""
    import json
    import subprocess
    import sys
    expected = set()
    for c in CASES.values():
        D, n_poly = dims(c["spec"])
        for _, family in c["paths"]:
            if family != "step":
                expected |= {instance(family, D, n_poly, j) for j in c["grads"]}
    assert len(ALL_INSTANCES) == 28 and expected == ALL_INSTANCES, sorted(ALL_INSTANCES - expected)
    print("measured maxima:", {k: "%.2e" % v for k, v in sorted(MEASURED.items())})
    env = {k: v for k, v in __import__("os").environ.items() if k not in ENV_VARS}
    script = _PROFILE_SCRIPT.replace("SYS_PATH", repr(sys.path)).replace("MODULE", __name__)
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", script]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    names = json.loads(r.stdout.strip().splitlines()[-1])
    for cid, c in CASES.items():
        D, n_poly = dims(c["spec"])
        for path, family in c["paths"]:
            for need_grad in c["grads"]:
                tag = "%s/%s/%s" % (cid, path, "grad" if need_grad else "nograd")
                check_kernels(set(names["%s|%s|%d" % (cid, path, need_grad)]), family, D, n_poly, need_grad, tag)
    if not any(PROFILED):
        pytest.skip("the profiler recorded no CUDA activity")
    print("reached:", sorted(REACHED))
    assert REACHED == ALL_INSTANCES, sorted(ALL_INSTANCES - REACHED)
