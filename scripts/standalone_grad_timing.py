"""Stand-alone policy forward + backward: the CUDA kernels (torch.ops.mcpilco.policy_forward, whose backward is
mcpilco_policy_backward) against torch autograd through oracle.policy_apply moved to the same GPU.

Shapes: C1 (cart-pole: M 400, nb 200, Dp 5, Du 1, angle policy), C4 (UR5: M 200, nb 400, Dp 24, Du 6, trajectory policy), and the C1
widths at M = 65 536 and 1 048 576.  Dropout p = 0.25 (Philox mask for the CUDA path, an injected mask for torch).  CUDA events around
`iters` forward + backward calls after `warmup` calls, median of 5 windows.  The inputs fit in L2 except at M = 1 048 576.

Flop count (FP64, an FMA counts 2, exp / tanh / Philox not counted), per particle and basis function:
  forward 4 Dp + 2 Du (distance, W h);  backward 4 Dp (distance again) + 6 Dp (d/dz, d/dc) + 4 Du (g_W, <la, W>) + 2 Du (squash sum)
so 14 Dp + 8 Du.  The share of peak is over the 34.15 TFLOP/s DFMA rate measured on this project's B200
(profiles/microbench/r02_fp64_peaks.txt).

usage: python scripts/standalone_grad_timing.py [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "mc-pilco_b200"))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

DFMA_PEAK = 34.15e12
SHAPES = [("C1", 400, 200, "angles", 1), ("C4", 200, 400, "target", 6), ("C1_M65536", 65536, 200, "angles", 1),
          ("C1_M1048576", 1048576, 200, "angles", 1)]


def flops(M, nb, Dp, Du):
    return float(M) * nb * (14 * Dp + 8 * Du)


def make(kind, M, nb, Du, dev, rs):
    from mcpilco_b200 import _pack as P
    from mcpilco_b200 import torch_ops as TO
    T = lambda a: torch.tensor(np.asarray(a), dtype=torch.float64, device=dev)  # noqa: E731
    if kind == "angles":
        Ds, Dp, extra = 4, 5, dict(angle=[2], non_angle=[0, 1, 3])
        x = T(rs.uniform(-2, 2, (M, Ds)))
        traj = None
    else:
        Ds, Dp, extra = 12, 24, {}
        traj = T(0.3 * rs.randn(4, Ds))
        x = traj[1] + T(0.3 * rs.randn(M, Ds))
    u_max = [10.0] * Du
    pst = P.policy_struct(kind, nb, Dp, Du, Ds, u_max=u_max, has_bias=False, use_drop=True, **extra)
    prm = {"log_ls": T(np.log(1.0 + rs.rand(1, Dp))), "centers": T(rs.uniform(-2, 2, (nb, Dp))), "W": T(rs.rand(Du, nb) - 0.5)}
    for v in prm.values():
        v.requires_grad_(True)
    x.requires_grad_(True)
    oracle = dict(kind=kind, bias=None, u_max=T(u_max), scale=T(np.ones((1, Dp))), target_traj=traj, **prm, **extra)
    return TO.policy_tensor(pst), prm, x, traj, oracle, Dp


def time_windows(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / iters)
    return float(np.median(out)), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "standalone_grad_timing.json"))
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("standalone_grad_timing: no CUDA device (this measurement has no CPU fallback)")
    from oracle import mcpilco_oracle as O
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    res = {"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip(), "p_dropout": 0.25, "dfma_peak_tflops": DFMA_PEAK / 1e12,
           "shapes": []}
    p = 0.25
    for name, M, nb, kind, Du in SHAPES:
        rs = np.random.RandomState(0)
        pt, prm, x, traj, oracle, Dp = make(kind, M, nb, Du, dev, rs)
        G = torch.randn(M, Du, dtype=torch.float64, device=dev)
        mask = (torch.rand(M, nb, device=dev) >= p).double()
        leaves = [prm["log_ls"], prm["centers"], prm["W"], x]

        def cuda_step():
            u = torch.ops.mcpilco.policy_forward(pt, prm["log_ls"], prm["centers"], prm["W"], None, traj, x, 1, p, None, 12345, 0)
            return torch.autograd.grad((u * G).sum(), leaves)

        def torch_step():
            u = O.policy_apply(oracle, x, 1, mask, p)
            return torch.autograd.grad((u * G).sum(), leaves)

        iters = 20 if M >= 1 << 20 else 100
        ms_cuda, w_cuda = time_windows(cuda_step, args.warmup, iters)
        ms_torch, w_torch = time_windows(torch_step, args.warmup, iters)
        fl = flops(M, nb, Dp, Du)
        row = {"shape": name, "M": M, "nb": nb, "Dp": Dp, "Du": Du, "cuda_ms": ms_cuda, "torch_autograd_ms": ms_torch,
               "speedup": ms_torch / ms_cuda, "flops": fl, "cuda_tflops": fl / (ms_cuda * 1e-3) / 1e12,
               "cuda_share_of_dfma_peak": fl / (ms_cuda * 1e-3) / DFMA_PEAK, "cuda_windows_ms": w_cuda, "torch_windows_ms": w_torch}
        res["shapes"].append(row)
        print(json.dumps({k: row[k] for k in ("shape", "M", "cuda_ms", "torch_autograd_ms", "speedup", "cuda_share_of_dfma_peak")}), flush=True)
        del mask, G, x, prm, oracle
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "nvidia_smi": res["nvidia_smi"]}))


if __name__ == "__main__":
    main()
