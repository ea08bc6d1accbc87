// Error-compensated INT8 tensor-core variant of the posterior contraction  V[M,N] = A[M,K] * B[N,K]^T  (A = K*, B = K^-1) —
// SURVEY.md §8 f4, the only route past the native FP64 pipe (37 TFLOP/s) on B200.  OPT-IN; the default path stays native fp64.
//
// Ozaki scheme I with exact integer slicing:
//   * each row of A (column of the product's right factor B) is scaled by a power of two 2^e so that |a| 2^-e < 1/4, converted to a
//     64-bit fixed-point integer F = rint(a 2^(8S - e)) and written as S balanced base-256 digits d_t in [-128, 127]
//     (a 2^-e = sum_t d_t 256^-(t+1), exact to 2^-8S);
//   * the product keeps the S(S+1)/2 digit-plane products with t + u < S:   A B^T = 2^(eA+eB) sum_w 256^-(w+2) C_w,
//     C_w = sum_{t+u=w} A_t B_u^T, every C_w an EXACT int32 GEMM (|C_w| <= (w+1) K 2^14 < 2^31 as long as S K <= 65536; a longer
//     contraction index is cut into segments that are recombined in fp64);
//   * A's planes are stored side by side along K and B's planes in REVERSE order, so C_w is one contraction with K_eff = (w+1) K over
//     contiguous sub-ranges of both operands;
//   * the plane sums are folded from the least significant up, in fp64, and the row / column scales applied last.
// The digit-plane products run on the 5th-generation tensor cores in ONE hand-written persistent kernel (ozaki_mma_kernel below:
// TMA -> tcgen05.mma.cta_group::2.kind::i8 -> int32 accumulators in TMEM -> tcgen05.ld -> fp64 recombination in the epilogue), so
// the int32 planes never exist in memory.  S = 8 carries 64 bits per entry (fp64-class results), S = 7 carries 56.  Measured accuracy
// and rates: DESIGN.md §4.
#include <cuda.h>

#include "mcp_common.cuh"

namespace mcp {

// ---- slicing: one warp per row -----------------------------------------------------------------------------------
// The contraction index is cut into `nseg` segments of Ks columns (S * Ks <= 65536 keeps every int32 plane product exact); a segment's
// planes are contiguous:  planes[row][seg][p][k],  p = t (reverse == 0) or S-1-t (reverse == 1), k < Ksp (Ks rounded up to 128, zero
// padded).  Row stride nseg * S * Ksp bytes.  One exponent per row, common to all segments; a row with a NaN or an infinity gets the
// exponent MCP_OZAKI_EXP_NONFINITE and zero digits, and the contraction's epilogue writes NaN wherever that row meets the product.
__global__ void __launch_bounds__(256) ozaki_slice_kernel(const double* __restrict__ A, int rows, int K, int ld, int S, int Ks, int Ksp, int nseg,
                                                          int reverse, int8_t* __restrict__ planes, int32_t* __restrict__ expo) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const double* a = A + (size_t)row * ld;
  double mx = 0.0;
  bool finite = true;
  for (int k = lane; k < K; k += 32) {
    const double v = a[k];
    finite = finite && isfinite(v);
    mx = fmax(mx, fabs(v));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  finite = __all_sync(0xffffffffu, finite);
  // |a| 2^-e < 1/4: the most significant balanced digit stays within [-65, 65] after the carries from below (no wrap at +128)
  const int e = !finite ? MCP_OZAKI_EXP_NONFINITE : mx > 0.0 ? ilogb(mx) + 3 : 0;
  if (lane == 0) expo[row] = e;
  int8_t* out = planes + (size_t)row * nseg * S * Ksp;
  const int sh = 8 * S - e;
  // four consecutive columns per lane: one packed 32-bit store per plane (Ksp is a multiple of 128, so groups never straddle a segment)
  for (int kk = lane * 4; kk < nseg * Ksp; kk += 128) {
    const int seg = kk / Ksp, k = kk - seg * Ksp, col = seg * Ks + k;
    long long F[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      F[i] = 0;
      if (finite && k + i < Ks && col + i < K) F[i] = __double2ll_rn(scalbn(a[col + i], sh));  // |F| < 2^(8S-2) <= 2^62
    }
    // balanced base-256 digits without a carry chain: F = sum_t d_t 256^t with d_t in [-128, 127]  <=>  F + sum_t 128 256^t has the
    // plain bytes d_t + 128, and (byte ^ 0x80) is d_t as int8.  Plane p holds digit t = S-1-p (most significant digit in plane 0).
    unsigned long long G[4];
    const unsigned long long bias = S >= 8 ? 0x8080808080808080ull : ((1ull << (8 * S)) - 1ull) / 255ull * 128ull;
#pragma unroll
    for (int i = 0; i < 4; i++) G[i] = ((unsigned long long)F[i] + bias) ^ bias;
    for (int p = 0; p < S; p++) {
      const int sh8 = 8 * (S - 1 - p);
      unsigned packed = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) packed |= ((unsigned)(G[i] >> sh8) & 255u) << (8 * i);
      *reinterpret_cast<unsigned*>(out + ((size_t)seg * S + (reverse ? S - 1 - p : p)) * Ksp + k) = packed;
    }
  }
}

// the persistent tcgen05 kernel (mcp_ozaki_mma.cu)
int ozaki_mma(const int8_t* Ap, const int32_t* Ae, const int8_t* Bp, const int32_t* Be, int M, int N, int S, int nseg, int Ksp, double* V, int ldv,
              cudaStream_t st);

// segmentation of the contraction index: nseg segments of Ks columns, Ksp = Ks rounded up to the MMA K tile
struct OzGeom {
  int nseg, Ks, Ksp;
};
static OzGeom ozaki_geom(int K, int S) {
  const int cap = 65536 / S / 128 * 128;  // S * Ks * 2^14 <= 2^30
  OzGeom g;
  g.nseg = (K + cap - 1) / cap;
  g.Ks = ((K + g.nseg - 1) / g.nseg + 127) / 128 * 128;
  if (g.Ks > cap) g.Ks = cap;
  g.nseg = (K + g.Ks - 1) / g.Ks;
  g.Ksp = g.Ks;
  return g;
}

// bytes of the digit planes of a [rows x K] matrix with S slices
void ozaki_geometry(int K, int S, int* nseg, int* Ks, int* Ksp) {
  const OzGeom g = ozaki_geom(K, S);
  *nseg = g.nseg;
  *Ks = g.Ks;
  *Ksp = g.Ksp;
}

size_t ozaki_plane_bytes(int rows, int K, int S) {
  const OzGeom g = ozaki_geom(K, S);
  return (size_t)rows * g.nseg * S * g.Ksp;
}

// scratch for one contraction of mc particles against N points: A's digit planes + A's exponents
size_t ozaki_scratch_bytes(int mc, int N, int S) {
  return align_up(ozaki_plane_bytes(mc, N, S), 256) + align_up((size_t)mc * 4, 256) + 1024;
}

int ozaki_slice(const double* A, int rows, int K, int ld, int S, int reverse, int8_t* planes, int32_t* expo, cudaStream_t st) {
  MCP_CHECK_ARG(S >= 2 && S <= 8, "ozaki: slices %d outside [2, 8]", S);
  if (rows <= 0) return MCP_OK;
  const OzGeom g = ozaki_geom(K, S);
  ozaki_slice_kernel<<<cdiv(rows, 8), 256, 0, st>>>(A, rows, K, ld, S, g.Ks, g.Ksp, g.nseg, reverse, planes, expo);
  MCP_LAUNCH_CHECK();
  return MCP_OK;
}

// V[mc, N] (fp64, ldv) = A[mc, N] (fp64, lda) * Binv^T given B's reversed digit planes / exponents
int ozaki_contract(const double* A, int lda, int mc, int N, int S, const int8_t* Bplanes, const int32_t* Bexp, double* V, int ldv, void* scratch,
                   size_t scratch_bytes, cudaStream_t st) {
  MCP_CHECK_ARG(scratch_bytes >= ozaki_scratch_bytes(mc, N, S), "ozaki: scratch too small");
  const OzGeom gm = ozaki_geom(N, S);
  char* p = (char*)align_up((size_t)scratch, 256);
  int8_t* Ap = (int8_t*)p; p += align_up(ozaki_plane_bytes(mc, N, S), 256);
  int32_t* Ae = (int32_t*)p;
  if (int e = ozaki_slice(A, mc, N, lda, S, 0, Ap, Ae, st)) return e;
  return ozaki_mma(Ap, Ae, Bplanes, Bexp, mc, N, S, gm.nseg, gm.Ksp, V, ldv, st);
}

}  // namespace mcp

using namespace mcp;

extern "C" __attribute__((visibility("default"))) int mcpilco_ozaki_available(void) { return 1; }

extern "C" __attribute__((visibility("default"))) size_t mcpilco_ozaki_plane_bytes(int N, int slices) { return ozaki_plane_bytes(N, N, slices); }

extern "C" __attribute__((visibility("default"))) int mcpilco_ozaki_prepare(const double* Kinv, int N, int ld, int slices, int8_t* planes,
                                                                             int32_t* exponents, void* stream) {
  MCP_CHECK_ARG(Kinv && planes && exponents && N >= 1 && ld >= N, "ozaki_prepare: bad arguments");
  return ozaki_slice(Kinv, N, N, ld, slices, 1, planes, exponents, (cudaStream_t)stream);
}

extern "C" __attribute__((visibility("default"))) size_t mcpilco_ozaki_scratch_bytes(int M, int N, int slices) { return ozaki_scratch_bytes(M, N, slices); }

extern "C" __attribute__((visibility("default"))) int mcpilco_ozaki_contract(const double* A, int lda, int M, int N, int slices, const int8_t* planes,
                                                                              const int32_t* exponents, double* V, int ldv, void* scratch,
                                                                              size_t scratch_bytes, void* stream) {
  MCP_CHECK_ARG(A && planes && exponents && V && scratch && M >= 1 && N >= 1 && lda >= N && ldv >= N, "ozaki_contract: bad arguments");
  return ozaki_contract(A, lda, M, N, slices, planes, exponents, V, ldv, scratch, scratch_bytes, (cudaStream_t)stream);
}
