#!/usr/bin/env python
"""bench.py — particle-steps/s of one GP particle rollout, forward + backward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # the CUDA path (mcpilco_b200)
    python bench.py --impl reference [--gpus N] [--steps K] ...     # the reference algorithm on the host CPU (oracle port)
    python bench.py --steps K --dump-outputs DIR                    # also write the last timed step's outputs, to compare two builds

A "step" is what one iteration of MC_PILCO.reinforce_policy does on the hot path (reference MC_PILCO.py:484-522):
apply_policy -> cost_function -> cost.backward(), i.e. M*H particle-steps forward and backward, including the cost, the
gradient reduction and (N > 1) the collectives.  Workload (config.workload): the "synthetic cartpole GP scaling sweep" point
N = 8192 training points, horizon 60, SE + polynomial kernel, E = 2 outputs, nb = 200 policy with dropout 0.25, M particles
PER GPU (weak scaling; 8 GPUs x 131072 is the north-star M = 1M — pass --particles-per-gpu 131072 for that; throughput per
particle-step does not depend on M beyond ~4k, see DESIGN.md).  Precompute (Cholesky etc.) is outside the metric and reported
in config.precompute_ms.  Nothing here reads /root/reference.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "mc-pilco_b200"))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FP64_PEAK_TFLOPS = 37.15  # measured on this pool's B200: DMMA.8x8x4 issue-bound, 3 s sustained (profiles/microbench/r01_fp64_peaks.txt)
METRIC = "particle-steps/s (rollout fwd+bwd)"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--train-points", type=int, default=8192)
    ap.add_argument("--particles-per-gpu", type=int, default=8192)
    ap.add_argument("--horizon", type=int, default=60)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-particles", type=int, default=512)
    ap.add_argument("--cpu-horizon", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cuda-profiler-range", action="store_true", help="cudaProfilerStart/Stop around the timed region (ncu --profile-from-start off)")
    ap.add_argument("--ozaki", type=int, default=0, choices=[0, 7, 8],
                    help="opt-in INT8 tensor-core contraction with error compensation for the main measurement (default 0: native fp64)")
    ap.add_argument("--no-variants", action="store_true", help="skip the extra timing of the opt-in INT8 contraction variants")
    ap.add_argument("--se-only", action="store_true", help="config 2 kernel (pure squared-exponential)")
    ap.add_argument("--no-real-shapes", action="store_true", help="skip the block that times BASELINE configs 1-4 at their real sizes")
    ap.add_argument("--no-forward-only", action="store_true", help="skip the forward-only (no-grad rollout) measurement")
    ap.add_argument("--cpu-particles-all", type=int, default=2048, help="cpu_baseline sample with all host threads: particles (SURVEY 8d: min(M, 2048))")
    ap.add_argument("--cpu-horizon-all", type=int, default=8, help="cpu_baseline sample with all host threads: horizon (SURVEY 8d: 8)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (states, inputs, cost, std, policy gradients) "
                         "as DIR/<name>.npy in float64; beyond 64 MB in all, states and inputs keep a seeded sample of the particles")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "own":
        ap.error("--dump-outputs dumps the CUDA path (--impl own)")
    return a


# ------------------------------------------------------------------------------------------------------------------
# CPU leg: the oracle port of the reference algorithm on the host cores (the only place bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------------------------
def cpu_rollout_sample(sc, M, H, threads, repeats, warmup, fitted=None):
    """Times `repeats` fwd+bwd rollouts of M particles x H steps with the oracle (torch CPU fp64, autograd) on the workload `sc`.
    `fitted`: optional [(alpha, Kinv)] per output (CPU tensors) to skip the O(N^3) fit, which is outside the metric."""
    from oracle import mcpilco_oracle as O
    torch.set_num_threads(threads)
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64)  # noqa: E731
    X = T(sc["X"])
    gps = []
    for e, g in enumerate(sc["gps"]):
        sp = O.make_spec(sc["D"], log_ls=g["log_ls"], log_lambda=float(np.log(g["lambda"])), mean=g["mean"],
                         mpk_log_pars=[np.log(w) for w in g["mpk"]], sigma_n=g["sigma_n"])
        if fitted is None:
            alpha, _, Kinv = O.gp_fit(sp, X, T(sc["Y"][:, e:e + 1]))
        else:
            alpha, Kinv = fitted[e]
        gps.append((sp, X, alpha, Kinv))
    m = dict(sc["model"]); m.update(Ds=sc["Ds"], Du=sc["Du"], norm=[1.0] * sc["E"])
    p = sc["policy"]
    rs = np.random.RandomState(1)
    times = []
    for it in range(warmup + repeats):
        pol = {"kind": p["kind"], "log_ls": T(np.log(p["lengthscales"])).reshape(1, -1).requires_grad_(True),
               "centers": T(p["centers"]).requires_grad_(True), "W": T(p["weight"]).requires_grad_(True), "bias": None,
               "u_max": p["u_max"], "scale": torch.ones(1, p["centers"].shape[1], dtype=torch.float64),
               "angle": list(p["angle"]), "non_angle": list(p["non_angle"])}
        eps0, eps = T(rs.randn(M, sc["Ds"])), T(rs.randn(H - 1, M, sc["E"]))
        masks = T((rs.rand(H, M, p["nb"]) >= sc["p_dropout"]).astype(np.float64))
        t0 = time.perf_counter()
        x0 = O.initial_particles(T(sc["x0_mean"]), T(sc["x0_var"]), eps0)
        st, inp = O.rollout(m, gps, pol, x0, eps, masks, sc["p_dropout"])
        c = sc["cost"]
        cost, std = O.expected_cost(O.cost_cart_pole(st, T(c["target"]), T(c["ls"]), c["angle_index"], c["pos_index"]))
        cost.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    return times


def cpu_fit(sc, threads):
    """[(alpha, Kinv)] per output from the oracle's own fit (reference GP_prior.py:91-115,130-135)."""
    from oracle import mcpilco_oracle as O
    torch.set_num_threads(threads)
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64)  # noqa: E731
    out = []
    for e, g in enumerate(sc["gps"]):
        sp = O.make_spec(sc["D"], log_ls=g["log_ls"], log_lambda=float(np.log(g["lambda"])), mean=g["mean"],
                         mpk_log_pars=[np.log(w) for w in g["mpk"]], sigma_n=g["sigma_n"])
        alpha, _, Kinv = O.gp_fit(sp, T(sc["X"]), T(sc["Y"][:, e:e + 1]))
        out.append((alpha, Kinv))
    return out


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0  # the CPU baseline is one process on rank 0
    from mcpilco_b200 import workloads as W
    sc = W.cartpole_sweep(args.train_points, se_only=args.se_only)
    cores = host_cores()
    M, H = args.cpu_particles, args.cpu_horizon
    fitted = cpu_fit(sc, cores)  # the O(N^3) fit is outside the metric: once, with all threads
    times = cpu_rollout_sample(sc, M, H, cores, args.steps, args.warmup, fitted=fitted)
    ms = 1e3 * float(np.sum(times))
    value = M * H * len(times) / float(np.sum(times))
    sample = "oracle port (torch CPU fp64 + autograd) of the same workload at M=%d particles x H=%d steps per step (memory ~ M*N*H*E forbids the full size), %d threads" % (M, H, cores)
    t1 = cpu_rollout_sample(sc, min(256, M), H, 1, repeats=1, warmup=0, fitted=fitted)
    one_thread = {"value": min(256, M) * H / float(np.sum(t1)), "unit": "particle-steps/s", "cores": 1,
                  "sample": "same port with torch.set_num_threads(1), the reference's shipped setting (test_mcpilco_cartpole.py:46-47), M=%d x H=%d, one rollout" % (min(256, M), H)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "particle-steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / max(len(times), 1), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, int(os.environ.get("WORLD_SIZE", "1"))),
            "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": cores, "kind": "port", "sample": sample, "one_thread": one_thread},
            "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0


def workload_config(args, world):
    return {"workload": "c5 synthetic cartpole GP sweep point: N=%d training points, M=%d particles/GPU (global %d), horizon %d, E=2, D=6, %s kernel, "
                        "nb=200 policy, p_dropout=0.25, Cart_pole_cost, Philox noise" % (args.train_points, args.particles_per_gpu,
                                                                                        args.particles_per_gpu * world, args.horizon,
                                                                                        "SE" if args.se_only else "SE+MPK(2)"),
            "train_points": args.train_points, "particles_per_gpu": args.particles_per_gpu, "horizon": args.horizon,
            "parallelism": "particle-dp%d" % world, "l2": "inputs larger than L2 (Kinv 2 x %d MB, K*/V chunks >= 1 GB)" % (args.train_points ** 2 * 8 >> 20)}


# ------------------------------------------------------------------------------------------------------------------
# CUDA arm
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi samples of one GPU while the timed region runs (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.path)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "power_w_max": max(power) if power else None, "samples": len(sm)}


def build_objects(sc, dev):
    """The reference's construction sequence (test_mcpilco_cartpole.py:49-231) against mcpilco_b200's classes."""
    import mcpilco_b200.model_learning.Model_learning as ML
    import mcpilco_b200.policy_learning.Cost_function as CF
    import mcpilco_b200.policy_learning.MC_PILCO as MCP
    import mcpilco_b200.policy_learning.Policy as PO
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)  # noqa: E731
    D = sc["D"]
    dicts = []
    for g in sc["gps"]:
        rbf = dict(active_dims=np.arange(D), lengthscales_init=np.exp(g["log_ls"]), lambda_init=np.array([g["lambda"]]), flg_train_lambda=False,
                   sigma_n_init=np.array([g["sigma_n"]]), dtype=torch.float64, device=dev)
        mpk = dict(active_dims=np.arange(D), poly_deg=len(g["mpk"]), Sigma_pos_par_init_list=list(g["mpk"]),
                   flg_train_Sigma_pos_par_list=[True] * len(g["mpk"]), dtype=torch.float64, device=dev)
        dicts.append([rbf, mpk] if g["mpk"] else rbf)
    m, p, c = sc["model"], sc["policy"], sc["cost"]
    cls = ML.Speed_Model_learning_RBF_MPK_angle_state if sc["gps"][0]["mpk"] else ML.Speed_Model_learning_RBF_angle_state
    model_par = dict(num_gp=sc["E"], init_dict_list=dicts, T_sampling=m["T"], angle_indeces=m["angle"], not_angle_indeces=m["not_angle"],
                     vel_indeces=m["vel"], not_vel_indeces=m["pos"], device=dev)
    policy_par = dict(state_dim=sc["Ds"], input_dim=sc["Du"], num_basis=p["nb"], angle_indices=p["angle"], non_angle_indices=p["non_angle"],
                      lengthscales_init=p["lengthscales"], centers_init=p["centers"], weight_init=p["weight"], flg_squash=True,
                      u_max=p["u_max"], flg_drop=True, device=dev)
    cost_par = dict(target_state=T(c["target"]), lengthscales=T(c["ls"]), angle_index=c["angle_index"], pos_index=c["pos_index"])
    obj = MCP.MC_PILCO(T_sampling=m["T"], state_dim=sc["Ds"], input_dim=sc["Du"], f_sim=None, f_model_learning=cls, model_learning_par=model_par,
                       f_rand_exploration_policy=None, rand_exploration_policy_par=None, f_control_policy=PO.Sum_of_gaussians_with_angles,
                       control_policy_par=policy_par, f_cost_function=CF.Cart_pole_cost, cost_function_par=cost_par, device=dev)
    ml = obj.model_learning
    ml.gp_inputs = T(sc["X"])
    ml.gp_output_list = [T(sc["Y"][:, e:e + 1]) for e in range(sc["E"])]
    ml.dim_state, ml.dim_input, ml.num_samples = sc["Ds"], sc["Du"], sc["N"]
    return obj


def real_shapes_block(dev, with_cpu):
    """BASELINE configs 1-4 at the reference's real sizes (SURVEY.md 8: C1-C4; latency-bound, ~1 GFLOP per rollout): per config the GPU
    time of one rollout forward + backward through the class API (CUDA events), the WALL time of one whole optimisation step of
    reinforce_policy's inner sequence (zero_grad, apply_policy, cost, the reference's NaN host sync of MC_PILCO.py:497, backward,
    torch Adam step) and, beside them, the oracle port of the reference on the host CPU (1 thread = the reference's shipped setting,
    test_mcpilco_cartpole.py:46-47, and all threads) on the same synthetic scenario."""
    from mcpilco_b200 import workloads as W
    import contextlib
    out = {}
    for key in W.REAL_SHAPES:
        sc = W.real_shape(key, with_noise=True)
        with contextlib.redirect_stdout(sys.stderr):
            obj = W.build_pilco(sc, dev)
        params = [p for p in obj.control_policy.parameters() if p.requires_grad]
        kw = W.apply_kwargs(sc, dev)
        opt = torch.optim.Adam(params, lr=1e-3)

        def fwd_bwd():
            for p in params:
                p.grad = None
            st, inp = obj.apply_policy(**kw)
            cost, _ = obj.cost_function(st, inp, 0)
            cost.backward()
            return cost

        def opt_step():
            opt.zero_grad(set_to_none=True)
            st, inp = obj.apply_policy(**kw)
            cost, _ = obj.cost_function(st, inp, 0)
            nan = bool(torch.isnan(cost))  # the per-step host synchronisation the reference's loop has
            cost.backward()
            opt.step()
            return nan

        reps = 10 if key == "c4" else 30
        for _ in range(3):
            fwd_bwd()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            cost = fwd_bwd()
        e1.record()
        torch.cuda.synchronize()
        gpu_ms = e0.elapsed_time(e1) / reps
        for _ in range(3):
            opt_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            opt_step()
        torch.cuda.synchronize()
        wall_ms = 1e3 * (time.perf_counter() - t0) / reps
        # the same step with the rollout's forward + backward captured in a CUDA graph (SURVEY.md 8 f1; what reinforce_policy runs)
        import mcpilco_b200.policy_learning.MC_PILCO as MCP
        graph_ms = graph_wall_ms = None
        if MCP._GraphedRollout.eligible(obj):
            obj._trial_index = 0
            init = dict(kw)
            p_drop = init.pop("p_dropout")
            g = MCP._GraphedRollout(obj, init, p_drop)

            def graph_step():
                c, _ = g.replay()
                nan = bool(torch.isnan(c))
                g.deposit_grads()
                opt.step()
                return nan

            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            graph_ms = e0.elapsed_time(e1) / reps
            for _ in range(3):
                graph_step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                graph_step()
            torch.cuda.synchronize()
            graph_wall_ms = 1e3 * (time.perf_counter() - t0) / reps
        row = {"N": sc["N"], "M": sc["M"], "H": sc["H"], "nb": sc["policy"]["nb"], "D": sc["D"], "E": sc["E"],
               "gpu_ms_fwd_bwd": gpu_ms, "opt_step_wall_ms": wall_ms, "wall_over_gpu": wall_ms / gpu_ms,
               "graph_gpu_ms_fwd_bwd": graph_ms, "graph_opt_step_wall_ms": graph_wall_ms,
               "particle_steps_per_s": sc["M"] * sc["H"] / ((graph_ms or gpu_ms) * 1e-3), "cost": float(cost.detach())}
        if with_cpu:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import helpers as Hh  # the oracle port of the reference: the CPU baseline leg only
            cores = host_cores()
            for label, thr in (("cpu_ms_1thread", 1), ("cpu_ms_all_threads", cores)):
                torch.set_num_threads(thr)
                gps = Hh.oracle_fit(sc)
                ts = []
                for it in range(1 if key == "c4" and thr == 1 else 2):
                    t0 = time.perf_counter()
                    Hh.oracle_rollout(sc, gps)
                    ts.append(time.perf_counter() - t0)
                row[label] = 1e3 * ts[-1]
            row["cpu_threads_all"] = cores
            row["speedup_vs_cpu_1thread"] = row["cpu_ms_1thread"] / (graph_ms or gpu_ms)
            row["speedup_vs_cpu_all_threads"] = row["cpu_ms_all_threads"] / (graph_ms or gpu_ms)
        out[key] = row
    return out


def own_arm(args):
    import torch.distributed as dist
    from mcpilco_b200 import _ops as ops
    from mcpilco_b200 import workloads as W
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device — the hot path has no CPU fallback")
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sc = W.cartpole_sweep(args.train_points, se_only=args.se_only)
    os.environ["MCPILCO_OZAKI"] = str(args.ozaki)
    obj = build_objects(sc, dev)
    ml, pol = obj.model_learning, obj.control_policy
    import contextlib
    pre_ms = []
    for _ in range(2):  # first pass: cold (module load, first allocations); second: what every later model update costs
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad(), contextlib.redirect_stdout(sys.stderr):
            for e in range(sc["E"]):
                ml.pretrain_gp(e)
        torch.cuda.synchronize()
        pre_ms.append(1e3 * (time.perf_counter() - t0))
    precompute_cold_ms, precompute_ms = pre_ms
    ml.set_eval_mode()
    M_global, H = args.particles_per_gpu * world, args.horizon
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)  # noqa: E731
    mean_d, var_d = T(sc["x0_mean"]), T(sc["x0_var"])
    kw = dict(flg_particles_init_uniform=False, particles_init_up_bound=None, particles_init_low_bound=None,
              flg_particles_init_multi_gauss=False, num_particles=M_global, T_control=H, p_dropout=sc["p_dropout"])
    params = [pol.log_lengthscales, pol.centers, pol.f_linear.weight]

    def step(mean=mean_d, var=var_d):
        for p in params:
            p.grad = None
        states, inputs = obj.apply_policy(particles_initial_state_mean=mean, particles_initial_state_var=var, **kw)
        cost, std = obj.cost_function(states, inputs, 0)
        cost.backward()
        return cost, std, states, inputs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    torch.manual_seed(0)
    for _ in range(args.warmup):
        step()
    # ---- timed region: inputs resident in HBM ----
    barrier()
    ops.prof_enable(True)
    ops.launch_count(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if args.cuda_profiler_range:
        torch.cuda.profiler.start()
    e0.record()
    for _ in range(args.steps):
        cost, std, states, inputs = step()
    e1.record()
    barrier()
    if args.cuda_profiler_range:
        torch.cuda.profiler.stop()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler is not None else None
    launches = ops.launch_count(reset=True)
    gemm_ms, gemm_n, gemm_fl = ops.prof_read()
    ops.prof_enable(False)
    cost_v = float(cost.detach())
    value = M_global * H * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:  # under torch.distributed: rank 0's particles
        dump_outputs(args.dump_outputs, {"states": states, "inputs": inputs, "cost": cost, "std_cost": std,
                                         "grad_log_lengthscales": pol.log_lengthscales.grad, "grad_centers": pol.centers.grad,
                                         "grad_weight": pol.f_linear.weight.grad}, per_particle=("states", "inputs"))
    del states, inputs  # not held through the measurements below

    # ---- end to end: host buffers in, host results out, through the same public API ----
    host_in = [p.detach().cpu().pin_memory() for p in params] + [mean_d.cpu().pin_memory(), var_d.cpu().pin_memory()]
    host_out = [torch.empty(n, dtype=torch.float64).pin_memory() for n in (2, pol.log_lengthscales.numel(), pol.centers.numel(), pol.f_linear.weight.numel())]
    h2d = sum(t.numel() * 8 for t in host_in)
    d2h = sum(t.numel() * 8 for t in host_out)

    def e2e_step():
        with torch.no_grad():
            for p, h in zip(params, host_in[:3]):
                p.copy_(h, non_blocking=True)
        mean = host_in[3].to(dev, non_blocking=True)
        var = host_in[4].to(dev, non_blocking=True)
        c, s = step(mean, var)[:2]
        host_out[0].copy_(torch.stack([c.detach(), s.detach()]), non_blocking=True)
        for h, p in zip(host_out[1:], params):
            h.copy_(p.grad.reshape(-1), non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the host reads the result

    ms_e2e, e2e_value = None, None
    if args.e2e_steps > 0:  # 0: skipped (the full north-star shard takes a minute per step; the default run always measures it)
        e2e_step()
        barrier()
        e0.record()
        for _ in range(args.e2e_steps):
            e2e_step()
        e1.record()
        barrier()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1))
        e2e_value = M_global * H * args.e2e_steps / (ms_e2e * 1e-3)

    # ---- opt-in variants of the dominant contraction (same workload, same API; reported beside the fp64 headline) ----
    variants = {}
    from mcpilco_b200 import _native as _Nn
    if not args.no_variants and args.ozaki == 0 and _Nn.lib().mcpilco_ozaki_available() and args.train_points >= 4096:
        REPLAY = 10 ** 6  # rollout counter -> Philox key: the same noise for the fp64 rollout and for each variant

        def replay_step():
            obj._rollouts = REPLAY
            c = step()[0]
            return float(c.detach()), [p.grad.detach().clone() for p in params]

        def grad_rel(ga, gb):
            return max(float((a - b).abs().max() / b.abs().max().clamp_min(1e-300)) for a, b in zip(ga, gb))

        c_ref, g_ref = replay_step()
        for S, tol in ((8, "posterior variance within 1e-7 relative of the fp64 path (tests/test_gpu_parity.py)"),
                       (7, "posterior variance within 1e-5 relative of the fp64 path")):
            os.environ["MCPILCO_OZAKI"] = str(S)
            ml._fitted_cache = None
            step(); step()
            barrier()
            ops.prof_enable(True)
            e0.record()
            for _ in range(2):
                vc = step()[0]
            e1.record()
            barrier()
            vms = max_over_ranks(e0.elapsed_time(e1)) / 2
            g_ms, g_n, g_fl = ops.prof_read()
            ops.prof_enable(False)
            c_var, g_var = replay_step()
            variants["ozaki%d" % S] = {"value": M_global * H / (vms * 1e-3), "unit": "particle-steps/s", "ms_per_step": vms, "cost": float(vc.detach()),
                                       "same_noise_vs_fp64": {"cost_rel_diff": abs(c_var - c_ref) / abs(c_ref), "policy_grad_rel_diff": grad_rel(g_var, g_ref),
                                                              "note": "one rollout + backward replayed with the fp64 run's Philox key (H = %d steps of error growth)" % H},
                                       "contraction": "int8 tcgen05 tensor cores, %d balanced base-256 digit planes per operand, int32 accumulation in TMEM, "
                                                      "fp64 recombination" % S,
                                       "contraction_tflops_fp64_equivalent": g_fl / (g_ms * 1e-3) * 1e-12 if g_ms > 0 else None,
                                       "tolerance": tol}
        os.environ["MCPILCO_OZAKI"] = "0"
        ml._fitted_cache = None

    # ---- forward-only rollout (no-grad: reference MC_PILCO.py:430-456, apply_mcpilco_policy_on_model.py:66-76): the contraction runs
    #      over the triangular factor L^-1 (N^2 flops per particle-step and output instead of 2 N^2) ----
    forward_only = None
    if not args.no_forward_only:
        def fwd_step():
            with torch.no_grad():
                st, inp = obj.apply_policy(particles_initial_state_mean=mean_d, particles_initial_state_var=var_d, **kw)
                return obj.cost_function(st, inp, 0)[0]
        fwd_step(); fwd_step()
        barrier()
        ops.prof_enable(True)
        e0.record()
        for _ in range(2):
            fc = fwd_step()
        e1.record()
        barrier()
        fms = max_over_ranks(e0.elapsed_time(e1)) / 2
        f_ms, f_n, f_fl = ops.prof_read()
        ops.prof_enable(False)
        Ns_ = [g.N for g in ml.fitted_gps()]
        Ff = W.flops_per_particle_step(Ns_, sc["D"], need_grad=False)
        fval = M_global * H / (fms * 1e-3)
        forward_only = {"value": fval, "unit": "particle-steps/s (rollout forward only)", "ms_per_step": fms, "cost": float(fc),
                        "flops_per_particle_step": Ff, "step_frac_of_fp64_peak": Ff * fval / world * 1e-12 / FP64_PEAK_TFLOPS,
                        "contraction": "w = K* L^-T over the triangle (dgemm_tma_kernel<TRIM>, heavy column tiles first), var = k** - |w|^2",
                        "contraction_tflops": f_fl / (f_ms * 1e-3) * 1e-12 if f_ms > 0 else None,
                        "contraction_frac_of_fp64_peak": f_fl / (f_ms * 1e-3) * 1e-12 / FP64_PEAK_TFLOPS if f_ms > 0 else None,
                        "kernel_share_of_step": f_ms / (2 * fms) if f_ms > 0 else None}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    Ns = [g.N for g in ml.fitted_gps()]
    F = W.flops_per_particle_step(Ns, sc["D"], need_grad=True)
    achieved = gemm_fl / (gemm_ms * 1e-3) * 1e-12 if gemm_ms > 0 else None
    traffic = None
    prof_json = os.path.join(ROOT, "profiles", "ncu_gemm_summary.json")
    if os.path.exists(prof_json):
        try:
            traffic = json.load(open(prof_json)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    line = {"metric": METRIC, "value": value, "unit": "particle-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64" if args.ozaki == 0 else "f64 results via int8 digit planes (Ozaki-%d)" % args.ozaki, "data": "synthetic",
            "config": dict(workload_config(args, world), precompute_ms=precompute_ms, precompute_cold_ms=precompute_cold_ms, cost=cost_v, e2e_steps=args.e2e_steps,
                           flops_per_particle_step=F, step_tflops_per_gpu=F * value / world * 1e-12,
                           step_frac_of_fp64_peak=F * value / world * 1e-12 / FP64_PEAK_TFLOPS,
                           # a rollout of H states has H - 1 GP transitions: the same fraction counted per transition
                           step_frac_of_fp64_peak_per_transition=F * value / world * 1e-12 / FP64_PEAK_TFLOPS * (H - 1) / H),
            "roofline": {"bound": "tensor", "kernel": ("dgemm_tma_kernel (V = K* Kinv, FP64 DMMA.8x8x4, TMA + mbarrier pipeline)" if args.ozaki == 0 else
                                                      "int8 tcgen05 plane GEMMs + slice/combine (fp64-equivalent flops)"), "achieved": achieved,
                         "peak": FP64_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": None if achieved is None else achieved / FP64_PEAK_TFLOPS,
                         "traffic": traffic,
                         "traffic_source": "STATIC: dram__bytes_read + dram__bytes_write of one launch from the committed ncu --set full capture "
                                           "(profiles/ncu_gemm_summary.json, M = N = 8192); not measured in this run — achieved/frac are live",
                         "launches_timed": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                         "flops_per_launch": gemm_fl / max(gemm_n, 1), "kernel_share_of_step": gemm_ms / ms,
                         "peak_source": "own measurement on this pool (FP64 is absent from MEASURED_PEAKS.json): profiles/microbench/r01_fp64_peaks.txt"},
            "e2e": {"value": e2e_value, "unit": "particle-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": None if ms_e2e is None else ms_e2e / args.e2e_steps},
            "gpu_launches": launches, "clocks": clocks, "variants": variants, "forward_only": forward_only}
    if world == 1 and not args.no_real_shapes:
        line["real_shapes"] = real_shapes_block(dev, with_cpu=not args.no_cpu_baseline)
    if world == 1 and not args.no_cpu_baseline:
        # SURVEY.md 8d: the sweep shape cannot be run by the reference at full size (memory ~ M N H E); all host threads at
        # min(M, 2048) x H = 8, and the reference's shipped single-thread setting on a smaller sample, both per particle-step
        cores = host_cores()
        fitted = [(g.alpha.detach().cpu().reshape(-1, 1), g.Kinv.detach().cpu().contiguous()) for g in ml.fitted_gps()]
        Ma, Ha = min(args.cpu_particles_all, args.particles_per_gpu), args.cpu_horizon_all
        cpu_rollout_sample(sc, 128, 2, cores, repeats=1, warmup=0, fitted=fitted)  # thread pool / allocator warm-up
        times = cpu_rollout_sample(sc, Ma, Ha, cores, repeats=1, warmup=0, fitted=fitted)
        M1, H1 = min(256, args.cpu_particles), args.cpu_horizon
        times1 = cpu_rollout_sample(sc, M1, H1, 1, repeats=1, warmup=0, fitted=fitted)
        line["cpu_baseline"] = {"value": Ma * Ha * len(times) / float(np.sum(times)), "unit": "particle-steps/s", "cores": cores, "kind": "port",
                                "sample": "oracle port (torch CPU fp64 + autograd; /root/reference cannot travel to the GPU box) of the same workload at "
                                          "M=%d x H=%d, one timed rollout after a small warm-up, %d threads" % (Ma, Ha, cores),
                                "one_thread": {"value": M1 * H1 / float(np.sum(times1)), "unit": "particle-steps/s", "cores": 1,
                                               "sample": "same port, torch.set_num_threads(1) (the reference's shipped setting, "
                                                         "test_mcpilco_cartpole.py:46-47), M=%d x H=%d, one rollout" % (M1, H1)}}
    emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, arrays, per_particle):
    """Write `arrays` (name -> tensor) as path/<name>.npy in float64.  The arrays named in `per_particle` are [H, M, ...]; when
    everything would exceed DUMP_BYTES they keep a seeded sample of the M particles (sorted, the same for each of them and for every
    run with the same M), so that dumps of two builds compare element for element."""
    out = {k: v.detach().double().cpu().numpy() for k, v in arrays.items()}
    M = out[per_particle[0]].shape[1]
    fixed = sum(a.nbytes for k, a in out.items() if k not in per_particle) + 128 * len(out)  # + the .npy headers
    per = sum(out[k].nbytes for k in per_particle) // M
    if fixed + M * per > DUMP_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(M, (DUMP_BYTES - fixed) // per, replace=False))
        for k in per_particle:
            out[k] = out[k][:, keep]
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a)


def emit(line):
    """The ONE JSON line of the contract, on the process's real stdout (see __main__)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

if __name__ == "__main__":
    a = parse()
    # stdout carries exactly one JSON line: everything else that writes to fd 1 — NCCL's version banner, library prints — goes to stderr
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    sys.exit(reference_arm(a) if a.impl == "reference" else own_arm(a))
