"""Exact host reference of the INT8 (Ozaki) contraction (mc-pilco_b200/csrc/mcp_ozaki.cu, mcp_ozaki_mma.cu).

Every step before the final scaling is integer-exact, so the device result is a deterministic function of the operands:

  * slice():     the digit planes and row exponents `ozaki_slice_kernel` writes (and `cov_slice_kernel`, given its exponents);
  * geometry():  the segmentation of the contraction index (`ozaki_geom`);
  * fold():      the plane sums C_w (exact: every partial sum is an integer below 2^31, so an fp64 matmul of the digit matrices is
                 exact in any summation order) folded in the epilogue's order, least significant first inside each segment and sweep,
                 each step one correctly rounded add of the exact product C_w 2^-8(w+2); then the row / column scale 2^(eA + eB).

numpy is used where the device arithmetic must be matched bit for bit (np.ldexp is exact and correctly rounded for any shift, unlike
torch.ldexp, which forms 2^e and overflows above 1023; np.rint rounds half to even like __double2ll_rn).
"""
import numpy as np

from mcpilco_b200 import _native

# exponent of a row that holds a non-finite entry (MCP_OZAKI_EXP_NONFINITE): its digits are zero and the contraction writes NaN to the
# whole row (A) or column (B) of V
EXP_NONFINITE = _native.OZAKI_EXP_NONFINITE
MMA_K = 128  # contraction bytes per k-block of the MMA kernel: segments are padded to a multiple of it


def geometry(K, S):
    """(nseg, Ks, Ksp) of ozaki_geom: nseg segments of Ks columns, S * Ks <= 65536 keeps every int32 plane sum exact."""
    cap = 65536 // S // MMA_K * MMA_K
    nseg = -(-K // cap)
    Ks = min((-(-K // nseg) + MMA_K - 1) // MMA_K * MMA_K, cap)
    nseg = -(-K // Ks)
    return nseg, Ks, Ks


def ilogb(x):
    """C ilogb of positive finite doubles, subnormals included (frexp normalises them: x = m 2^q with m in [0.5, 1))."""
    return np.frexp(x)[1].astype(np.int64) - 1


def row_exponents(a):
    """ozaki_slice_kernel's row exponents: ilogb(max |a|) + 3 (so |a| 2^-e < 1/4), 0 for a zero row, EXP_NONFINITE for a row with a
    NaN or an infinity."""
    a = np.asarray(a, dtype=np.float64)
    fin = np.isfinite(a).all(axis=1)
    mx = np.where(np.isfinite(a), np.abs(a), 0.0).max(axis=1) if a.shape[1] else np.zeros(a.shape[0])
    e = np.where(mx > 0, ilogb(np.where(mx > 0, mx, 1.0)) + 3, 0)
    return np.where(fin, e, EXP_NONFINITE).astype(np.int64)


def fixed_point(a, S, e):
    """F = rint(a 2^(8S - e)) per entry (int64); zero in rows marked non-finite."""
    a = np.asarray(a, dtype=np.float64)
    e = np.asarray(e, dtype=np.int64)
    bad = e == EXP_NONFINITE
    sh = np.where(bad, 0, 8 * S - e)[:, None]
    x = np.rint(np.ldexp(np.where(bad[:, None], 0.0, a), sh))
    return x.astype(np.int64)


def digits(F, S):
    """Balanced base-256 digits d_t in [-128, 127] with F = sum_t d_t 256^t, t = 0 least significant; returned [..., S] as int8,
    formed the way the kernels form them: the bytes of (F + sum_t 128 256^t) ^ (sum_t 128 256^t)."""
    bias = np.uint64(0x8080808080808080 if S >= 8 else ((1 << (8 * S)) - 1) // 255 * 128)
    G = (np.ascontiguousarray(F).astype("<u8") + bias) ^ bias
    return G.view(np.int8).reshape(F.shape + (8,))[..., :S]  # little-endian: byte t is digit t


def slice(a, S, reverse, e=None):
    """Digit planes (int8 [rows, nseg, S, Ksp]) and exponents (int64 [rows]) of the rows of a [rows, K], laid out as
    ozaki_slice_kernel writes them: planes[row][seg][p][k], plane p = digit S-1-p (most significant first), in reverse plane order
    for reverse=1 (the right factor), columns past K zero.  e given: slice with these row exponents (cov_slice_kernel)."""
    a = np.asarray(a, dtype=np.float64)
    rows, K = a.shape
    nseg, Ks, Ksp = geometry(K, S)
    e = row_exponents(a) if e is None else np.asarray(e, dtype=np.int64)
    F = np.zeros((rows, nseg * Ks), dtype=np.int64)
    F[:, :K] = fixed_point(a, S, e)
    d = digits(F, S).reshape(rows, nseg, Ks, S)[..., ::-1]       # [..., p]: plane p = digit S-1-p
    if reverse:
        d = d[..., ::-1]
    planes = np.zeros((rows, nseg, S, Ksp), dtype=np.int8)
    planes[:, :, :, :Ks] = np.moveaxis(d, -1, 2)
    return planes, e


def edge_rows(K, S, rs):
    """Rows where slicing goes wrong: zeros, a single nonzero, a maximum of exactly 2^k and just below, rint ties, a subnormal
    maximum, a maximum near DBL_MAX, 1e-200 next to 1, and plain random rows with a row scale from 1e-3 to 1e3."""
    rows = [np.zeros(K)]
    r = np.zeros(K)
    r[rs.randint(K)] = -3.7
    rows.append(r)
    for top in (2.0 ** 5, np.nextafter(2.0 ** 5, 0.0), -2.0 ** -7):
        r = rs.uniform(-1, 1, K) * abs(top)
        r[rs.randint(K)] = top
        rows.append(r)
    # ties (2j+1) 2^(e - 8S - 1) of a row whose maximum 1.5 gives the exponent e = ilogb(1.5) + 3: |2j+1| < 2^(8S-2) keeps them below
    # the maximum at every S, and below 2^51 so that 2j+1 is exact in fp64
    e, lim = 3, 2 ** min(8 * S - 3, 50)
    r = (2.0 * rs.randint(-lim, lim, K) + 1.0) * 2.0 ** (e - 8 * S - 1)
    r[rs.randint(K)] = 1.5
    rows.append(r)
    rows.append(rs.uniform(-1, 1, K) * 2.0 ** -1060)                  # subnormal maximum
    r = rs.uniform(-1, 1, K) * 1e307
    r[rs.randint(K)] = -np.finfo(np.float64).max * 0.999
    rows.append(r)
    r = np.where(rs.rand(K) < 0.5, 1e-200, rs.uniform(-1, 1, K))
    r[rs.randint(K)] = 1.0
    rows.append(r)
    for s in np.logspace(-3, 3, 4):
        rows.append(rs.randn(K) * s)
    return np.stack(rows)


def sweeps(S):
    """Plane-sum indices w of the epilogue's sweeps in fold order: sweep 0 = S-1 .. max(0, S-4), sweep 1 = S-5 .. 0."""
    out = [list(range(S - 1, max(0, S - 4) - 1, -1))]
    if S > 4:
        out.append(list(range(S - 5, -1, -1)))
    return out


def fold(Ap, eA, Bp, eB, S, device="cpu"):
    """V [M, N] (numpy float64) from A's planes (forward order) and B's planes (reversed), exactly as the MMA kernel's epilogue
    forms it.  The plane sums are fp64 matmuls of the digit matrices on `device` (exact); non-finite-marked rows / columns are NaN."""
    import torch
    M, nseg, _, Ksp = Ap.shape
    N = Bp.shape[0]
    A = torch.as_tensor(np.ascontiguousarray(Ap)).to(device)
    B = torch.as_tensor(np.ascontiguousarray(Bp)).to(device)
    v = torch.zeros(M, N, dtype=torch.float64, device=device)
    for seg in range(nseg):
        for ws in sweeps(S):
            for w in ws:
                # C_w = sum_{t+u=w} A_t B_u^T: A's planes 0..w side by side against B's digits w..0 (stored reversed: planes S-1-w..S-1)
                a = A[:, seg, :w + 1, :].reshape(M, -1).double()
                b = B[:, seg, S - 1 - w:, :].reshape(N, -1).double()
                v = v + (a @ b.t()) * 2.0 ** (-8 * (w + 2))
    v = v.cpu().numpy()
    eA, eB = np.asarray(eA, dtype=np.int64), np.asarray(eB, dtype=np.int64)
    bad = (eA[:, None] == EXP_NONFINITE) | (eB[None, :] == EXP_NONFINITE)
    with np.errstate(over="ignore"):  # a row maximum near DBL_MAX may scale to inf, as on the device
        return np.where(bad, np.nan, np.ldexp(v, np.where(bad, 0, eA[:, None] + eB[None, :])))


def reference(A, B, S, device="cpu"):
    """(V, A's planes and exponents, B's planes and exponents) of the contraction A [M, K] @ B [N, K]^T with S digit planes."""
    Ap, eA = slice(A, S, 0)
    Bp, eB = slice(B, S, 1)
    return fold(Ap, eA, Bp, eB, S, device), Ap, eA, Bp, eB
