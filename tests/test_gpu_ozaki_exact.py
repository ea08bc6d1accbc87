"""The opt-in INT8 (Ozaki) contraction bit for bit against the exact host reference (tests/ozaki_ref.py).

Before the last scaling every step of the scheme is integer-exact and the epilogue fixes the fold order, so the digit planes, the row
exponents and V are deterministic functions of the operands: every comparison here is equality, no tolerance.  Covered:

  * slicing (mcpilco_ozaki_prepare and the A side of mcpilco_ozaki_contract): every byte of the plane buffers, padding included, and
    every exponent, for S = 2 .. 8 and edge rows (zeros, a single nonzero, maxima at and just below a power of two, rint ties, a
    subnormal maximum, a maximum near DBL_MAX, 1e-200 next to 1);
  * the contraction over plane counts 2 .. 8 (S outside {7, 8} runs the MMA issuer's run-time schedule, S <= 4 the one-sweep layout with
    double-buffered slots), tile edges of the 256 x 128 pair tiles, 289 tiles (several per cluster, a short last raster group), two
    segments of the contraction index, leading dimensions larger than N with NaN padding that must be neither read nor written;
  * the posterior paths of mcpilco_gp_predict: every cov_slice_kernel<DT, NP> instance (K* rows, exponents from the Cauchy-Schwarz
    bound, digit planes, V), the non-fused path (wide inputs, a kernel without an SE term), particle chunking;
  * non-finite operands: a NaN / inf in a row of A gives a NaN row of V, one in a row of K^-1 a NaN column.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as Hh
import ozaki_ref as R

pytestmark = pytest.mark.gpu

F64 = torch.float64
NAN = float("nan")
PAD = -1234.5678  # finite sentinel in V's padding columns: the contraction writes NaN for marked rows, so NaN could not show a stray write


def _lib():
    from mcpilco_b200 import _native as Nn
    L = Nn.lib()
    if not L.mcpilco_ozaki_available():
        pytest.skip("built without CUTLASS headers")
    return L, Nn.check


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _al(x):
    return (x + 255) // 256 * 256


def ld16(n):
    return (n + 15) // 16 * 16


def padded(X, ld):
    """X [rows, n] in a [rows, ld] device buffer whose columns n.. hold NaN."""
    buf = torch.full((X.shape[0], ld), NAN, dtype=F64, device="cuda")
    buf[:, :X.shape[1]] = torch.as_tensor(X, dtype=F64)
    return buf


def prepare(Bbuf, N, S):
    """mcpilco_ozaki_prepare into device buffers pre-filled with 0xA5 / a junk exponent; returns (planes uint8, exponents int32)."""
    L, check = _lib()
    planes = torch.full((L.mcpilco_ozaki_plane_bytes(N, S),), 0xA5, dtype=torch.uint8, device="cuda")
    pexp = torch.full((N,), -77777, dtype=torch.int32, device="cuda")
    check(L.mcpilco_ozaki_prepare(_p(Bbuf), N, Bbuf.stride(0), S, _p(planes), _p(pexp), _st()))
    return planes, pexp


def scratch_planes(buf, base_off, rows, N, S):
    """A's digit planes and exponents as the contraction lays them out in its scratch (mcp_ozaki.cu, ozaki_contract): planes at the
    first 256-byte boundary, exponents at the next one after them.  buf: host bytes of the scratch, base_off: byte offset of the
    scratch pointer's 256-aligned start."""
    nseg, Ks, Ksp = R.geometry(N, S)
    nb = rows * nseg * S * Ksp
    planes = buf[base_off:base_off + nb].view(np.int8).reshape(rows, nseg, S, Ksp)
    expo = buf[base_off + _al(nb):base_off + _al(nb) + 4 * rows].view(np.int32).astype(np.int64)
    return planes, expo


def contract(Abuf, M, N, S, planes, pexp, ldv):
    """mcpilco_ozaki_contract with a scratch the test keeps: returns V (host, [M, ldv], pre-filled PAD) and A's planes / exponents."""
    L, check = _lib()
    sb = L.mcpilco_ozaki_scratch_bytes(M, N, S)
    scratch = torch.full((sb,), 0xA5, dtype=torch.uint8, device="cuda")
    V = torch.full((M, ldv), PAD, dtype=F64, device="cuda")
    check(L.mcpilco_ozaki_contract(_p(Abuf), Abuf.stride(0), M, N, S, _p(planes), _p(pexp), _p(V), ldv, _p(scratch), sb, _st()))
    Ap, Ae = scratch_planes(scratch.cpu().numpy(), (-scratch.data_ptr()) % 256, M, N, S)
    return V.cpu().numpy(), Ap, Ae


def check_contraction(A, B, S, lda=None, ldb=None, ldv=None):
    """Slice B (prepare) and contract A against it; planes, exponents and V must equal the reference exactly, and the padding columns
    of V (pre-filled with a finite sentinel) must keep it."""
    A, B = np.asarray(A, dtype=np.float64), np.asarray(B, dtype=np.float64)
    M, N = A.shape
    lda, ldb, ldv = lda or N + 3, ldb or N + 5, ldv or ld16(N)
    planes, pexp = prepare(padded(B, ldb), N, S)
    V, Ap, Ae = contract(padded(A, lda), M, N, S, planes, pexp, ldv)
    rBp, rBe = R.slice(B, S, 1)
    rAp, rAe = R.slice(A, S, 0)
    assert np.array_equal(pexp.cpu().numpy(), rBe), "B exponents"
    assert np.array_equal(planes.cpu().numpy().view(np.int8), rBp.reshape(-1)), "B planes"
    assert np.array_equal(Ae, rAe), "A exponents"
    assert np.array_equal(Ap, rAp), "A planes"
    ref = R.fold(rAp, rAe, rBp, rBe, S, device="cuda")
    bad = ~((V[:, :N] == ref) | (np.isnan(V[:, :N]) & np.isnan(ref)))
    assert not bad.any(), ("V differs from the exact fold", int(bad.sum()), np.argwhere(bad)[:5].tolist())
    assert (V[:, N:] == PAD).all(), "V padding written"
    return V[:, :N], ref


def operands(M, N, seed):
    """The row / column scalings of the fp64 parity test: A's rows from 1e-3 to 1e3, B's rows from 1e2 to 1e-2."""
    rs = np.random.RandomState(seed)
    A = rs.randn(M, N) * np.logspace(-3, 3, M)[:, None]
    B = rs.randn(N, N) * np.logspace(2, -2, N)[:, None]
    return A, B


# ---------------------------------------------------------------------------------------------------------------------
# slicing
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [1, 127, 128, 129, 8193])
@pytest.mark.parametrize("S", range(2, 9))
def test_prepare_planes_and_exponents_exact(S, N):
    rs = np.random.RandomState(7 * N + S)
    B = rs.randn(N, N) * np.logspace(-3, 3, N)[:, None]
    edges = R.edge_rows(N, S, rs)
    k = min(N, edges.shape[0])
    B[:k] = edges[:k]
    planes, pexp = prepare(padded(B, N + 3), N, S)
    rBp, rBe = R.slice(B, S, 1)
    assert np.array_equal(pexp.cpu().numpy(), rBe)
    got = planes.cpu().numpy().view(np.int8)
    assert got.size == rBp.size and np.array_equal(got, rBp.reshape(-1)), int((got != rBp.reshape(-1)).sum())


@pytest.mark.parametrize("S", range(2, 9))
def test_contract_slices_edge_rows_of_a_exactly(S):
    """A's slicing inside mcpilco_ozaki_contract (forward plane order) on the edge rows, then V."""
    rs = np.random.RandomState(S)
    N = 129
    A = np.concatenate([R.edge_rows(N, S, rs), R.edge_rows(N, S, rs)[::-1]])
    B = rs.randn(N, N)
    check_contraction(A, B, S)


# ---------------------------------------------------------------------------------------------------------------------
# contraction
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", range(2, 9))
def test_contraction_every_plane_count(S):
    A, B = operands(300, 257, S)
    check_contraction(A, B, S)


@pytest.mark.parametrize("N", [1, 16, 17, 63, 64, 65, 129])
@pytest.mark.parametrize("M", [1, 127, 128, 129, 256, 257])
@pytest.mark.parametrize("S", [8, 5, 3])
def test_contraction_tile_edges(S, M, N):
    A, B = operands(M, N, 1000 * S + M + N)
    check_contraction(A, B, S)


@pytest.mark.parametrize("S", [8, 5])
def test_contraction_many_tiles(S):
    """(4097, 2049): 17 x 17 = 289 pair tiles, several per cluster, and a last raster group of one tile row."""
    A, B = operands(4097, 2049, S)
    check_contraction(A, B, S)


@pytest.mark.parametrize("N,S", [(8192, 8), (8193, 8), (9344, 7), (9345, 7)])
def test_contraction_segment_boundary(N, S):
    """One segment at N = 65536 / S rounded down to 128 columns, two one column later."""
    A, B = operands(300, N, N)
    assert R.geometry(N, S)[0] == (1 if N % 2 == 0 else 2)
    check_contraction(A, B, S)


@pytest.mark.parametrize("M,N", [(129, 65), (300, 257), (1, 17), (257, 129)])
@pytest.mark.parametrize("ldv", ["N", "N+1", "ld16"])
def test_contraction_leading_dimensions(M, N, ldv):
    """ldv = N with odd N (rows not 16-byte aligned: the epilogue's scalar path), N + 1 and ld16(N); lda > N with NaN padding."""
    A, B = operands(M, N, M + N)
    check_contraction(A, B, 8, lda=N + 1, ldv={"N": N, "N+1": N + 1, "ld16": ld16(N)}[ldv])


@pytest.mark.parametrize("M", [1, 129, 300])
def test_contraction_c1_kinv(M):
    """B = K^-1 of the cart-pole C1 model (cond_1 ~ 1.8e6), A = rows of K* scale."""
    g = Hh.load_golden("c1")
    B = np.asarray(g["Kinv_0"], dtype=np.float64)
    rs = np.random.RandomState(M)
    A = np.abs(rs.randn(M, B.shape[0])) * np.exp(-rs.rand(M, B.shape[0]) * 8)
    for S in (8, 7, 5):
        check_contraction(A, B, S)


# ---------------------------------------------------------------------------------------------------------------------
# non-finite operands
# ---------------------------------------------------------------------------------------------------------------------
def test_contraction_nonfinite_rows_and_columns():
    """A NaN / inf in row m of A makes row m of V NaN, one in row n of B column n; everything else equals the exact fold."""
    _lib()
    A, B = operands(300, 257, 3)
    A[3, 100], A[7, 0], A[299, 256] = np.nan, np.inf, -np.inf
    B[2, 5], B[10, 256], B[256, 1] = -np.inf, np.nan, np.inf
    for S in (8, 7, 3):
        V, _ = check_contraction(A, B, S)
        rows, cols = np.isnan(V).all(1), np.isnan(V).all(0)
        assert list(np.nonzero(rows)[0]) == [3, 7, 299] and list(np.nonzero(cols)[0]) == [2, 10, 256]
        assert not np.isnan(V[~rows][:, ~cols]).any()
    from mcpilco_b200 import _ops as ops
    V, _, pexp = ops.ozaki_matmul(torch.as_tensor(A, device="cuda"), torch.as_tensor(B, device="cuda"), 8)
    fp64 = torch.as_tensor(A, device="cuda") @ torch.as_tensor(B, device="cuda").t()
    assert torch.equal(torch.isnan(V), ~torch.isfinite(fp64))
    assert (pexp.cpu().numpy()[[2, 10, 256]] == R.EXP_NONFINITE).all()


# ---------------------------------------------------------------------------------------------------------------------
# posterior paths (mcpilco_gp_predict with a workspace the test owns)
# ---------------------------------------------------------------------------------------------------------------------
def gp_spec(D, n_poly, se=True, seed=0):
    from mcpilco_b200 import _pack as P
    rs = np.random.RandomState(seed + 10 * D + n_poly)
    mpk = [np.exp(rs.uniform(-5, -3, D + 1)), np.exp(rs.uniform(-5, -2, 2 * D))][:n_poly]
    return P.spec_from_dict({"D": D, "log_ls": rs.uniform(0.0, 1.5, D) if se else None, "lambda": 1.7, "mean": 0.0, "mpk": mpk,
                             "sigma_n": 0.1})


_fits = {}


@pytest.fixture(scope="module", autouse=True)
def _release_device_memory():
    """Give the module's cached fits and the allocator's blocks back when the module is done."""
    yield
    _fits.clear()
    torch.cuda.empty_cache()


def fitted(D, n_poly, se, N, S):
    """A fitted GP (own precompute) on a random training set, with S planes of K^-1 prepared; cached per shape."""
    from mcpilco_b200 import _ops as ops
    key = (D, n_poly, se, N)
    if key not in _fits:
        spec = gp_spec(D, n_poly, se)
        rs = np.random.RandomState(N + D)
        X = torch.as_tensor(rs.uniform(-2, 2, (N, D)), device="cuda")
        y = torch.as_tensor(np.sin(rs.randn(N, 1)), device="cuda")
        alpha, Kinv = ops.gp_precompute(spec, X, y)
        _fits[key] = (spec, X, alpha, Kinv)
    spec, X, alpha, Kinv = _fits[key]
    return spec, X, ops.FittedGp(spec, X, alpha, Kinv, ozaki_slices=S)


def particles(X, M, seed):
    """M test inputs scattered around the training set."""
    rs = np.random.RandomState(seed)
    Xn = X.cpu().numpy()
    Xs = Xn[rs.randint(0, Xn.shape[0], M)] + 0.3 * rs.randn(M, Xn.shape[1])
    return Xs


def predict(gp, Xs, jac, ws_bytes=None):
    """mcpilco_gp_predict through ctypes; returns the outputs and the host bytes of the workspace with its 256-aligned start."""
    from mcpilco_b200 import _ops as ops
    L, check = _lib()
    Xs = torch.as_tensor(Xs, dtype=F64, device="cuda").contiguous()
    M, D = Xs.shape
    wsb = ws_bytes or workspace_bytes(gp.N, gp.ozaki, M)
    ws = torch.full((wsb,), 0xA5, dtype=torch.uint8, device="cuda")
    out = [torch.empty(M, 1, dtype=F64, device="cuda") for _ in range(2)]
    out += [torch.empty(M, 1, D, dtype=F64, device="cuda") for _ in range(2)] if jac else [None, None]
    arr = ops._gp_array([gp])
    check(L.mcpilco_gp_predict(arr, 1, _p(Xs), M, *[_p(t) for t in out], _p(ws), wsb, _st()))
    torch.cuda.synchronize()
    return out, ws.cpu().numpy(), (-ws.data_ptr()) % 256, wsb


def per_particle(N, S):
    """Workspace doubles per particle of gp_posterior_chunk on the INT8 path (mcp_gp.cu): K* and V rows, K*'s planes and exponent."""
    L, _ = _lib()
    return 2 * ld16(N) + (L.mcpilco_ozaki_scratch_bytes(1024, N, S) // 1024 + 7) // 8 + 1


def workspace_bytes(N, S, Mc):
    """A workspace that holds exactly Mc particles per chunk, whatever the alignment of its start."""
    return 8 * (16384 + Mc * per_particle(N, S)) + 255


def chunk_rows(N, S, nbytes, off, M):
    """Particles per chunk of gp_posterior_chunk for a workspace of nbytes whose 256-aligned start is off bytes in."""
    return min(((nbytes - off) // 8 - 16384) // per_particle(N, S), M)


def posterior_layout(buf, off, M, Mc, N, S):
    """K* [M, ld16(N)], V [M, ld16(N)] and K*'s digit planes / exponents of the last chunk (M rows) in the workspace: K* at the
    256-aligned start, V after Mc rows, the planes at the next 256-byte boundary after 2 Mc rows."""
    ldk = ld16(N)
    f = buf[off:off + 16 * Mc * ldk].view(np.float64)
    Ks = f[:M * ldk].reshape(M, ldk)
    V = f[Mc * ldk:Mc * ldk + M * ldk].reshape(M, ldk)
    return Ks, V, *scratch_planes(buf, off + 16 * Mc * ldk, M, N, S)


COV_SLICE = {f"cov_slice_kernel<{dt}, {npl}>" for dt in (4, 6, 8) for npl in (0, 1, 2)} - {"cov_slice_kernel<8, 2>"}
# (D, n_poly, has SE, N): every cov_slice_kernel<DT, NP> instance, and (fused = False) the non-fused path
POSTERIOR = [(3, 0, True, 300), (4, 1, True, 257), (2, 2, True, 129), (5, 0, True, 300), (6, 1, True, 300), (6, 2, True, 1000),
             (7, 0, True, 300), (8, 1, True, 300), (6, 2, True, 8300), (24, 0, True, 300), (4, 2, False, 300)]


def fused_of(D, n_poly, se):
    return se and D <= 8 and not (D > 6 and n_poly == 2)


@pytest.mark.parametrize("jac", [True, False])
@pytest.mark.parametrize("S", [8, 7])
@pytest.mark.parametrize("D,n_poly,se,N", POSTERIOR)
def test_posterior_ozaki_path_exact(D, n_poly, se, N, S, jac):
    """K* equals gp_covariance; on the fused path its exponents equal max(ilogb(sqrt(k(x,x) kdiag_max) (1 + 1e-9)) + 3, -900) and
    bound every entry (|K*| 2^-e < 1/4), on the non-fused path they are the slicer's; the planes equal the reference slice of the K*
    row the kernel wrote, K^-1's planes the reference slice of K^-1, and V the exact fold."""
    from mcpilco_b200 import _ops as ops
    spec, X, gp = fitted(D, n_poly, se, N, S)
    M = 300
    Xs = particles(X, M, N + S)
    Xs[0] = X[int(ops.gp_diag_covariance(spec, X).argmax())].cpu().numpy()  # |K*| meets the Cauchy-Schwarz bound here
    out, buf, off, wsb = predict(gp, Xs, jac)
    fused = fused_of(D, n_poly, se)
    assert chunk_rows(N, S, wsb, off, M) == M
    Ks, V, Ap, Ae = posterior_layout(buf, off, M, M, N, S)
    Xt = torch.as_tensor(Xs, device="cuda")
    Kref = ops.gp_covariance(spec, Xt, X).cpu().numpy()
    assert np.array_equal(Ks[:, :N], Kref) and not Ks[:, N:].any()
    if fused:
        kd = ops.gp_diag_covariance(spec, Xt).cpu().numpy()
        bound = np.sqrt(kd * gp.kdiag_max) * (1.0 + 1e-9)
        ok = (bound > 0) & np.isfinite(bound)
        e = np.where(ok, np.maximum(R.ilogb(np.where(ok, bound, 1.0)) + 3, -900), 0)
        assert np.array_equal(Ae, e)
        assert (np.ldexp(np.abs(Kref), -e[:, None]) < 0.25).all()
        rAp, _ = R.slice(Kref, S, 0, e=e)
    else:
        rAp, e = R.slice(Kref, S, 0)
        assert np.array_equal(Ae, e)
    assert np.array_equal(Ap, rAp)
    rBp, rBe = R.slice(gp.Kinv.cpu().numpy(), S, 1)
    assert np.array_equal(gp.plane_exp.cpu().numpy(), rBe) and np.array_equal(gp.planes.cpu().numpy().view(np.int8), rBp.reshape(-1))
    ref = R.fold(rAp, e, rBp, rBe, S, device="cuda")
    assert np.array_equal(V[:, :N], ref), int((V[:, :N] != ref).sum())
    m0 = ops.gp_predict([ops.FittedGp(spec, X, gp.alpha, gp.Kinv, ozaki_slices=0)], Xt, jac=jac)[0]
    assert torch.equal(out[0], m0)  # the mean does not go through the contraction


@pytest.mark.parametrize("D,n_poly,se", [(6, 2, True), (24, 0, True)])
def test_posterior_chunks_bit_identical(D, n_poly, se):
    """A workspace for 100 particles per chunk: M = 350 runs as 100 + 100 + 100 + 50, bit-identical to the single-chunk call."""
    spec, X, gp = fitted(D, n_poly, se, 300, 8)
    M, N, S = 350, 300, 8
    Xs = particles(X, M, 5)
    one, *_ = predict(gp, Xs, True)
    wsb = workspace_bytes(N, S, 100)
    chunked, buf, off, _ = predict(gp, Xs, True, ws_bytes=wsb)
    assert chunk_rows(N, S, wsb, off, M) == 100
    for a, b in zip(one, chunked):
        assert torch.equal(a, b)
    # the workspace holds the last chunk (particles 300 .. 349): the split really happened
    from mcpilco_b200 import _ops as ops
    Ks, *_ = posterior_layout(buf, off, 50, 100, N, S)
    assert np.array_equal(Ks[:, :N], ops.gp_covariance(spec, torch.as_tensor(Xs[300:], device="cuda"), X).cpu().numpy())


@pytest.mark.parametrize("D,n_poly,se", [(6, 2, True), (24, 0, True)])
def test_posterior_nonfinite(D, n_poly, se):
    """A NaN particle gives NaN mean and variance (its K* row is NaN) and leaves the others bit-identical; a K^-1 with a NaN row gives
    NaN variances exactly where the fp64 path does, with the mean unchanged."""
    from mcpilco_b200 import _ops as ops
    spec, X, gp = fitted(D, n_poly, se, 300, 8)
    Xs = particles(X, 64, 9)
    base, *_ = predict(gp, Xs, True)
    Xs[5] = np.nan
    got, *_ = predict(gp, Xs, True)
    assert torch.isnan(got[0][5]).all() and torch.isnan(got[1][5]).all()
    keep = [i for i in range(64) if i != 5]
    for a, b in zip(base, got):
        assert torch.equal(a[keep], b[keep])
    Xs[5] = Xs[6]
    Kinv = gp.Kinv.clone()
    Kinv[7] = NAN
    Xt = torch.as_tensor(Xs, device="cuda")
    for S in (8, 7):
        m8, v8, _, jv8 = ops.gp_predict([ops.FittedGp(spec, X, gp.alpha, Kinv, ozaki_slices=S)], Xt, jac=True)
        m0, v0, _, jv0 = ops.gp_predict([ops.FittedGp(spec, X, gp.alpha, Kinv, ozaki_slices=0)], Xt, jac=True)
        assert torch.isnan(v0).any() and torch.equal(torch.isnan(v8), torch.isnan(v0)) and torch.equal(torch.isnan(jv8), torch.isnan(jv0))
        assert torch.equal(m8, m0) and torch.isfinite(m8).all()


def expected_kernels(D, n_poly, se):
    dt = 4 if D <= 4 else 6 if D <= 6 else 8
    return {"ozaki_mma_kernel", f"cov_slice_kernel<{dt}, {n_poly}>" if fused_of(D, n_poly, se) else "ozaki_slice_kernel"}


_PROFILE_CASES = r"""
import json, sys
sys.path[:0] = %r
import torch
from torch.profiler import ProfilerActivity, profile
import %s as T
names = {}
for D, n_poly, se, N in T.POSTERIOR:
    spec, X, gp = T.fitted(D, n_poly, se, min(N, 300), 8)
    Xs = T.particles(X, 64, 1)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        T.predict(gp, Xs, True)
        torch.cuda.synchronize()
    names[repr((D, n_poly, se))] = sorted({ev.name for ev in prof.events()})
print(json.dumps(names))
"""


def test_every_kernel_is_reached():
    """The posterior cases above reach the intended kernels: each fused case its cov_slice_kernel<DT, NP> instance and no other, each
    non-fused case ozaki_slice_kernel, all of them ozaki_mma_kernel; together all eight cov_slice_kernel instances.  The profiler runs
    in a child process so that its CUDA activity tracing cannot outlive this test."""
    import json
    import subprocess
    import sys
    _lib()
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _PROFILE_CASES % (sys.path, __name__)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    names = json.loads(r.stdout.strip().splitlines()[-1])
    if not any(names.values()):
        pytest.skip("the profiler recorded no CUDA activity")
    reached = set()
    for D, n_poly, se, N in POSTERIOR:
        got = {k for k in COV_SLICE | {"ozaki_mma_kernel", "ozaki_slice_kernel"} if any(k in nm for nm in names[repr((D, n_poly, se))])}
        assert got == expected_kernels(D, n_poly, se), (D, n_poly, se, sorted(got))
        reached |= got
    assert len(COV_SLICE) == 8 and reached == COV_SLICE | {"ozaki_mma_kernel", "ozaki_slice_kernel"}, sorted(reached)
