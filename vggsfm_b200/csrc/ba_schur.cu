// Schur-complement reduce, reduced-system preparation and back-substitution kernels.
//
// Replaces the Ceres SchurEliminator + DENSE_SCHUR/SPARSE_SCHUR Cholesky that
// pycolmap.bundle_adjustment runs on the host (vggsfm/utils/triangulation.py:1050,1142).
//
//   point_prep      per point: V = Dp H_pp Dp + diag(clamp(diag))/radius, 3x3 Cholesky,
//                   M = Dp L^-T, q = M^T g_p
//   assemble_hc     camera Hessian/gradient from the per-frame records into the dense reduced system
//   z_build         Zt[3n+c][row] = (W[n][row][:] M_n)[c]   (k-major operand for the SYRK; W is track-major,
//                   so this is a straight streaming pass), rhs[row] += Z[row] . q
//   (SYRK)          Sraw -= Zt^T Zt on the lower-triangular 128x128 tiles: tcgen05 INT8 Ozaki slices, csrc/syrk_i8.cu
//   scale_damp      A = Dc Sraw Dc + diag(clamp(diag(Dc Hcc Dc)))/radius, constant parameters pinned
//   cam_step / backsub_partial / point_step / cam_update   back-substitution and the candidate state
#include <stddef.h>
#include "common.cuh"

namespace vgg {

// band structure of the running solve (csrc/ba_solve.cu, compute_band_hint); null pointers: dense
BandDev g_band_dev = {nullptr, nullptr, nullptr, 0};

// Add v to one element of the reduced-system buffer.  Single GPU: plain f64 RED on the local copy.  Track-sharded
// multi-GPU ("fabric" mode): ONE multimem reduction on the NVSwitch multicast address, which lands the addend in every
// rank's copy of the buffer -- the all-reduce of the reduced camera system happens inside the kernels that
// produce it (assemble, z_build, SYRK epilogue), tile by tile, instead of in a separate NCCL call afterwards.
__device__ __forceinline__ void ar_add(double* local, double* mc, double v) {
  if (mc) asm volatile("multimem.red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(mc), "d"(v) : "memory");
  else atomicAdd(local, v);
}
__device__ __forceinline__ void ar_put(double* local, double* mc, double v) {   // buffer is zero beforehand
  if (mc) asm volatile("multimem.red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(mc), "d"(v) : "memory");
  else *local = v;
}

// ------------------------------------------------------------------------------------------------
__global__ void jacobi_scale_points_kernel(int N, const double* __restrict__ H_pp, double* __restrict__ sc_p, int enable) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const double* h = H_pp + (size_t)n * 6;
  sc_p[n * 3 + 0] = enable ? 1.0 / (1.0 + sqrt(h[0])) : 1.0;
  sc_p[n * 3 + 1] = enable ? 1.0 / (1.0 + sqrt(h[3])) : 1.0;
  sc_p[n * 3 + 2] = enable ? 1.0 / (1.0 + sqrt(h[5])) : 1.0;
}

__global__ void jacobi_scale_cams_kernel(int D, const double* __restrict__ hdiag, double* __restrict__ sc_c, int enable) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= D) return;
  sc_c[i] = enable ? 1.0 / (1.0 + sqrt(hdiag[i])) : 1.0;
}

// ------------------------------------------------------------------------------------------------
// per point: M (3x3 row-major) = Dp L^-T, q = M^T g_p, dpp = clamped scaled diagonal
__global__ void point_prep_kernel(int N, const double* __restrict__ H_pp, const double* __restrict__ g_p,
                                  const double* __restrict__ sc_p, const uint8_t* __restrict__ point_const,
                                  double radius, double min_diag, double max_diag, double* __restrict__ M,
                                  double* __restrict__ q, double* __restrict__ dpp, double* __restrict__ scal) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  double* Mo = M + (size_t)n * 9;
  if (point_const && point_const[n]) {
#pragma unroll
    for (int i = 0; i < 9; ++i) Mo[i] = 0.0;
    q[n * 3] = q[n * 3 + 1] = q[n * 3 + 2] = 0.0;
    dpp[n * 3] = dpp[n * 3 + 1] = dpp[n * 3 + 2] = 0.0;
    return;
  }
  const double* h = H_pp + (size_t)n * 6;
  const double s0 = sc_p[n * 3], s1 = sc_p[n * 3 + 1], s2 = sc_p[n * 3 + 2];
  double v00 = h[0] * s0 * s0, v01 = h[1] * s0 * s1, v02 = h[2] * s0 * s2;
  double v11 = h[3] * s1 * s1, v12 = h[4] * s1 * s2, v22 = h[5] * s2 * s2;
  const double d0 = fmin(fmax(v00, min_diag), max_diag);
  const double d1 = fmin(fmax(v11, min_diag), max_diag);
  const double d2 = fmin(fmax(v22, min_diag), max_diag);
  dpp[n * 3] = d0; dpp[n * 3 + 1] = d1; dpp[n * 3 + 2] = d2;
  v00 += d0 / radius; v11 += d1 / radius; v22 += d2 / radius;
  // Cholesky V = L L^T
  bool bad = !(v00 > 0.0);
  const double l00 = sqrt(v00);
  const double l10 = v01 / l00, l20 = v02 / l00;
  const double t11 = v11 - l10 * l10;
  bad = bad || !(t11 > 0.0);
  const double l11 = sqrt(t11);
  const double l21 = (v12 - l20 * l10) / l11;
  const double t22 = v22 - l20 * l20 - l21 * l21;
  bad = bad || !(t22 > 0.0);
  const double l22 = sqrt(t22);
  if (bad) {
    atomicAdd(&scal[6], 1.0);
#pragma unroll
    for (int i = 0; i < 9; ++i) Mo[i] = 0.0;
    q[n * 3] = q[n * 3 + 1] = q[n * 3 + 2] = 0.0;
    return;
  }
  // Linv (lower)
  const double i00 = 1.0 / l00, i11 = 1.0 / l11, i22 = 1.0 / l22;
  const double i10 = -l10 * i00 * i11;
  const double i21 = -l21 * i11 * i22;
  const double i20 = -(l20 * i00 + l21 * i10) * i22;
  // M = Dp Linv^T : M[r][c] = s_r * Linv[c][r]
  const double m00 = s0 * i00, m01 = s0 * i10, m02 = s0 * i20;
  const double m11 = s1 * i11, m12 = s1 * i21;
  const double m22 = s2 * i22;
  Mo[0] = m00; Mo[1] = m01; Mo[2] = m02;
  Mo[3] = 0.0; Mo[4] = m11; Mo[5] = m12;
  Mo[6] = 0.0; Mo[7] = 0.0; Mo[8] = m22;
  const double g0 = g_p[n * 3], g1 = g_p[n * 3 + 1], g2 = g_p[n * 3 + 2];
  q[n * 3 + 0] = m00 * g0;
  q[n * 3 + 1] = m01 * g0 + m11 * g1;
  q[n * 3 + 2] = m02 * g0 + m12 * g1 + m22 * g2;
}

// ------------------------------------------------------------------------------------------------
// camera records -> dense reduced system (both triangles of the diagonal blocks and borders),
// rhs = -g, hdiag, gvec.  One CTA per frame, plus one for the shared-intrinsics block.
__global__ void assemble_hc_kernel(int S, int dc, int ns, int KR, int Dpad, const double* __restrict__ camrec,
                                   const double* __restrict__ shared_in, double* __restrict__ Sraw,
                                   double* __restrict__ rhs, double* __restrict__ hdiag, double* __restrict__ gvec,
                                   ptrdiff_t mc_off) {
  const int s = blockIdx.x;
  const int tid = threadIdx.x;
#define VGG_PUT(ptr, val) ar_put((ptr), mc_off ? (ptr) + mc_off : nullptr, (val))
  if (s < S) {
    const double* rec = camrec + (size_t)s * KR;
    const int base = s * dc;
    if (tid < dc) {
      VGG_PUT(&gvec[base + tid], rec[tid]);
      VGG_PUT(&rhs[base + tid], -rec[tid]);
    }
    if (tid < dc * dc) {
      const int i = tid / dc, j = tid % dc;
      const int a = i < j ? i : j, b = i < j ? j : i;
      const int idx = dc + a * dc - a * (a - 1) / 2 + (b - a);
      const double val = rec[idx];
      VGG_PUT(&Sraw[(size_t)(base + i) * Dpad + base + j], val);
      if (i == j) VGG_PUT(&hdiag[base + i], val);
    }
    if (tid < 6 * ns) {
      const int i = tid / ns, j = tid % ns;
      const double val = rec[dc + dc * (dc + 1) / 2 + tid];
      VGG_PUT(&Sraw[(size_t)(S * dc + j) * Dpad + base + i], val);
      VGG_PUT(&Sraw[(size_t)(base + i) * Dpad + S * dc + j], val);
    }
  } else if (ns > 0) {
    const int base = S * dc;
    if (tid < ns) {
      VGG_PUT(&gvec[base + tid], shared_in[tid]);
      VGG_PUT(&rhs[base + tid], -shared_in[tid]);
    }
    if (tid < ns * ns) {
      const int i = tid / ns, j = tid % ns;
      const int a = i < j ? i : j, b = i < j ? j : i;
      const double val = shared_in[2 + (a == 0 ? b : 2)];
      VGG_PUT(&Sraw[(size_t)(base + i) * Dpad + base + j], val);
      if (i == j) VGG_PUT(&hdiag[base + i], val);
    }
  }
#undef VGG_PUT
}

// ------------------------------------------------------------------------------------------------
// Schur operand: Zt[(3n+c)*Dpad + row] = sum_c' W[n][row][c'] M[n][c'][c];  rhs[row] += sum_{n,c} Z q.
// W is track-major ([N][pitch][3]), so for a fixed track both the read (24 B per row) and the three writes
// (8 B per row into three k-rows of Zt) are contiguous across threads: no transpose, no shared-memory tile.
// block = 128 rows x ZB_NT tracks.
constexpr int ZB_NT = 32;
__global__ void __launch_bounds__(128) z_build_kernel(int D, int N, int Dpad, size_t pitch, const double* __restrict__ W,
                                                      const double* __restrict__ M, const double* __restrict__ q,
                                                      double* __restrict__ Zt, double* __restrict__ rhs,
                                                      ptrdiff_t mc_off, unsigned long long* __restrict__ amax,
                                                      const int* __restrict__ rb_range) {
  __shared__ double sm[ZB_NT][12];
  const int row = blockIdx.x * 128 + threadIdx.x;
  const int n0 = blockIdx.y * ZB_NT;
  const int nt = min(ZB_NT, N - n0);
  // banded problems: these 32 tracks' rows of Zt lie outside the k range in which this 128-column block is non-zero --
  // W is zero here (never written after the per-solve memset), nobody reads this part of Zt, nothing to add to rhs
  if (rb_range) {
    const int kb_first = (3 * n0) >> 6, kb_last = (3 * (n0 + nt - 1) + 2) >> 6;
    if (kb_last < rb_range[2 * blockIdx.x] || kb_first >= rb_range[2 * blockIdx.x + 1]) return;
  }
  for (int e = threadIdx.x; e < nt * 12; e += 128) {
    const int t = e / 12, k = e % 12;
    sm[t][k] = k < 9 ? M[(size_t)(n0 + t) * 9 + k] : q[(size_t)(n0 + t) * 3 + (k - 9)];
  }
  __syncthreads();
  if (row >= D) return;
  double zq = 0.0;
  double zmax = 0.0;                  // running max |z| of this row (NaN / Inf stick): the tensor-core SYRK's column scale
  const double* wp = W + ((size_t)n0 * pitch + row) * 3;
#pragma unroll 4
  for (int t = 0; t < nt; ++t, wp += pitch * 3) {
    const double w0 = wp[0], w1 = wp[1], w2 = wp[2];
    const double* m = sm[t];
    const double z0 = w0 * m[0];                              // M upper triangular (row-major)
    const double z1 = w0 * m[1] + w1 * m[4];
    const double z2 = w0 * m[2] + w1 * m[5] + w2 * m[8];
    double* zo = Zt + (size_t)(3 * (n0 + t)) * Dpad + row;
    zo[0] = z0;
    zo[Dpad] = z1;
    zo[2 * (size_t)Dpad] = z2;
    zq += z0 * m[9] + z1 * m[10] + z2 * m[11];
    const double a0 = fabs(z0), a1 = fabs(z1), a2 = fabs(z2);
    zmax = (a0 > zmax || a0 != a0) ? a0 : zmax;
    zmax = (a1 > zmax || a1 != a1) ? a1 : zmax;
    zmax = (a2 > zmax || a2 != a2) ? a2 : zmax;
  }
  if (amax) {
    if (!(zmax <= 1.7976931348623157e308)) zmax = __longlong_as_double(0x7ff0000000000000LL);
    if (zmax > 0.0) atomicMax(&amax[row], (unsigned long long)__double_as_longlong(zmax));
  }
  if (zq != 0.0) ar_add(&rhs[row], mc_off ? &rhs[row] + mc_off : nullptr, zq);
}

// ------------------------------------------------------------------------------------------------
// A (in place) = sc_i sc_j Sraw + diag; constant parameters pinned; b = sc * rhs.  Lower triangle only.
__global__ void scale_damp_kernel(int D, int Dpad, double* __restrict__ A, const double* __restrict__ rhs,
                                  const double* __restrict__ hdiag, const double* __restrict__ sc,
                                  const uint8_t* __restrict__ pconst, double radius, double min_diag, double max_diag,
                                  double* __restrict__ bvec) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  const int i = blockIdx.y;
  if (j > i) return;
  const bool ci = pconst[i] != 0, cj = pconst[j] != 0;
  double v;
  if (ci || cj) {
    v = (i == j) ? 1.0 : 0.0;
  } else {
    v = A[(size_t)i * Dpad + j] * sc[i] * sc[j];
    if (i == j) v += fmin(fmax(hdiag[i] * sc[i] * sc[i], min_diag), max_diag) / radius;
  }
  A[(size_t)i * Dpad + j] = v;
  if (i == j) {
    // The scaled right-hand side also becomes row D of the matrix (in the workspace rhs IS row D, so this scales it in
    // place): the factorisation of the bordered
    // matrix [[A, b], [b^T, c]] = [[L, 0], [y^T, .]] leaves y = L^-1 b there, i.e. the forward substitution comes out
    // of the factorisation for free (csrc/ba_solve.cu).  c only has to exceed y^T y.
    const double b = ci ? 0.0 : rhs[i] * sc[i];
    bvec[i] = b;
    A[(size_t)D * Dpad + i] = b;
    if (i == 0) A[(size_t)D * Dpad + D] = 1e300;
  }
}

// d_c = sc * dcs ; scal[0] += sum dcs^2 dcc/r (free) - d_c.g ; scal[1] += |d_c|^2 ; scal[7] non-finite flag
__global__ void cam_step_kernel(int D, const double* __restrict__ dcs, size_t dcs_stride, const double* __restrict__ sc,
                                const double* __restrict__ hdiag, const double* __restrict__ gvec,
                                const uint8_t* __restrict__ pconst, double radius, double min_diag, double max_diag,
                                double* __restrict__ d_c, double* __restrict__ scal) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double a = 0, b = 0, bad = 0;
  if (i < D) {
    const double x = pconst[i] ? 0.0 : dcs[(size_t)i * dcs_stride];
    const double dc = x * sc[i];
    d_c[i] = dc;
    if (!isfinite(x)) bad = 1.0;
    const double dcc = fmin(fmax(hdiag[i] * sc[i] * sc[i], min_diag), max_diag);
    a = pconst[i] ? 0.0 : (x * x * dcc / radius - dc * gvec[i]);
    b = dc * dc;
  }
  a = warp_sum(a); b = warp_sum(b); bad = warp_sum(bad);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&scal[0], a);
    atomicAdd(&scal[1], b);
    if (bad > 0) atomicAdd(&scal[7], bad);
  }
}

// wacc[n][c] = sum_row W[n][row][c] d_c[row]: one warp per track, lanes stride over the contiguous rows
__global__ void __launch_bounds__(256) backsub_kernel(int D, int N, size_t pitch, const double* __restrict__ W,
                                                      const double* __restrict__ d_c, double* __restrict__ wacc,
                                                      const int* __restrict__ kb_rows, int arrow_row) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (n >= N) return;
  const double* wp = W + (size_t)n * pitch * 3;
  double w0 = 0, w1 = 0, w2 = 0;
  auto span = [&](int r0, int r1) {
#pragma unroll 4
    for (int r = r0 + lane; r < r1; r += 32) {
      const double d = __ldg(d_c + r);
      w0 = fma(wp[(size_t)r * 3], d, w0);
      w1 = fma(wp[(size_t)r * 3 + 1], d, w1);
      w2 = fma(wp[(size_t)r * 3 + 2], d, w2);
    }
  };
  if (kb_rows) {
    // banded problems: the rows this point can touch (its two k-blocks' row ranges) and the dense arrow
    const int ka = (3 * n) >> 6, kb = (3 * n + 2) >> 6;
    const int lo = min(kb_rows[2 * ka], kb_rows[2 * kb]), hi = min(max(kb_rows[2 * ka + 1], kb_rows[2 * kb + 1]), arrow_row);
    if (lo < hi) span(lo, hi);
    span(min(arrow_row, D), D);
  } else {
    span(0, D);
  }
  w0 = warp_sum(w0); w1 = warp_sum(w1); w2 = warp_sum(w2);
  if (lane == 0) {
    wacc[(size_t)n * 3] = w0;
    wacc[(size_t)n * 3 + 1] = w1;
    wacc[(size_t)n * 3 + 2] = w2;
  }
}

// d_p = M M^T (-(g_p + w)); candidate = X + d_p; scal[2] += sum dps^2 dpp/r - d_p.g_p; scal[3] += |d_p|^2
__global__ void point_step_kernel(int N, const double* __restrict__ M, const double* __restrict__ g_p,
                                  const double* __restrict__ wacc, const double* __restrict__ sc_p,
                                  const double* __restrict__ dpp, const double* __restrict__ X, double radius,
                                  double* __restrict__ Xc, double* __restrict__ scal) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  double a = 0, b = 0;
  if (n < N) {
    const double* m = M + (size_t)n * 9;
    const double g0 = g_p[n * 3], g1 = g_p[n * 3 + 1], g2 = g_p[n * 3 + 2];
    const double y0 = -(g0 + wacc[n * 3]), y1 = -(g1 + wacc[n * 3 + 1]), y2 = -(g2 + wacc[n * 3 + 2]);
    // t = M^T y (M upper triangular)
    const double t0 = m[0] * y0;
    const double t1 = m[1] * y0 + m[4] * y1;
    const double t2 = m[2] * y0 + m[5] * y1 + m[8] * y2;
    const double d0 = m[0] * t0 + m[1] * t1 + m[2] * t2;
    const double d1 = m[4] * t1 + m[5] * t2;
    const double d2 = m[8] * t2;
    Xc[n * 3] = X[n * 3] + d0;
    Xc[n * 3 + 1] = X[n * 3 + 1] + d1;
    Xc[n * 3 + 2] = X[n * 3 + 2] + d2;
    const double s0 = sc_p[n * 3], s1 = sc_p[n * 3 + 1], s2 = sc_p[n * 3 + 2];
    const double e0 = d0 / s0, e1 = d1 / s1, e2 = d2 / s2;
    a = (e0 * e0 * dpp[n * 3] + e1 * e1 * dpp[n * 3 + 1] + e2 * e2 * dpp[n * 3 + 2]) / radius -
        (d0 * g0 + d1 * g1 + d2 * g2);
    b = d0 * d0 + d1 * d1 + d2 * d2;
  }
  a = warp_sum(a); b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&scal[2], a);
    atomicAdd(&scal[3], b);
  }
}

// candidate cameras: R <- Exp(2 delta) R, t <- t + dt, intrinsics
__global__ void cam_update_kernel(int S, int dc, int ns, int model, const double* __restrict__ d_c,
                                  const double* __restrict__ poses, const double* __restrict__ intr,
                                  double* __restrict__ poses_c, double* __restrict__ intr_c) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= S) return;
  const double* d = d_c + (size_t)s * dc;
  const double p0 = 2.0 * d[0], p1 = 2.0 * d[1], p2 = 2.0 * d[2];
  const double th2 = p0 * p0 + p1 * p1 + p2 * p2;
  const double th = sqrt(th2);
  double a, b;
  if (th < 1e-12) {
    a = 1.0 - th2 / 6.0;
    b = 0.5 - th2 / 24.0;
  } else {
    a = sin(th) / th;
    b = (1.0 - cos(th)) / th2;
  }
  // E = I + a K + b K^2
  double E[9];
  E[0] = 1.0 + b * (-(p1 * p1 + p2 * p2)); E[1] = -a * p2 + b * p0 * p1;           E[2] = a * p1 + b * p0 * p2;
  E[3] = a * p2 + b * p0 * p1;             E[4] = 1.0 + b * (-(p0 * p0 + p2 * p2)); E[5] = -a * p0 + b * p1 * p2;
  E[6] = -a * p1 + b * p0 * p2;            E[7] = a * p0 + b * p1 * p2;            E[8] = 1.0 + b * (-(p0 * p0 + p1 * p1));
  const double* P = poses + (size_t)s * 12;
  double* Q = poses_c + (size_t)s * 12;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) Q[i * 4 + j] = E[i * 3] * P[j] + E[i * 3 + 1] * P[4 + j] + E[i * 3 + 2] * P[8 + j];
  Q[3] = P[3] + d[3];
  Q[7] = P[7] + d[4];
  Q[11] = P[11] + d[5];
  const int ni = (model == VGG_SIMPLE_PINHOLE) ? 1 : 2;
  double f = intr[s * 4], k = intr[s * 4 + 3];
  if (dc > 6) {
    f += d[6];
    if (ni > 1) k += d[7];
  } else if (ns > 0) {
    const double* dsh = d_c + (size_t)S * dc;
    f += dsh[0];
    if (ni > 1) k += dsh[1];
  }
  intr_c[s * 4] = f;
  intr_c[s * 4 + 1] = intr[s * 4 + 1];
  intr_c[s * 4 + 2] = intr[s * 4 + 2];
  intr_c[s * 4 + 3] = k;
}

// gradient of the candidate camera block out of its records
__global__ void extract_gvec_kernel(int S, int dc, int ns, int KR, const double* __restrict__ camrec,
                                    const double* __restrict__ shared_in, double* __restrict__ gvec) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int D = S * dc + ns;
  if (i >= D) return;
  gvec[i] = (i < S * dc) ? camrec[(size_t)(i / dc) * KR + (i % dc)] : shared_in[i - S * dc];
}

// scal[4] = max |gvec| over free parameters, scal[5] = max |g_p| over variable points
__global__ void gradmax_kernel(int D, int N, const double* __restrict__ gvec, const uint8_t* __restrict__ pconst,
                               const double* __restrict__ g_p, const uint8_t* __restrict__ point_const,
                               double* __restrict__ scal) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  double mc = 0, mp = 0;
  if (i < D && !pconst[i]) mc = fabs(gvec[i]);
  if (i < N * 3 && !(point_const && point_const[i / 3])) mp = fabs(g_p[i]);
  mc = warp_max(mc); mp = warp_max(mp);
  if ((threadIdx.x & 31) == 0) {
    // non-negative doubles order like their bit patterns
    atomicMax(reinterpret_cast<unsigned long long*>(&scal[4]), (unsigned long long)__double_as_longlong(mc));
    atomicMax(reinterpret_cast<unsigned long long*>(&scal[5]), (unsigned long long)__double_as_longlong(mp));
  }
}

// ------------------------------------------------------------------------------------------------
// host-side launch helpers used by ba_solve.cu
// ------------------------------------------------------------------------------------------------
int launch_jacobi_scale_points(int N, const double* H_pp, double* sc_p, int enable, cudaStream_t st) {
  jacobi_scale_points_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, H_pp, sc_p, enable);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_jacobi_scale_cams(int D, const double* hdiag, double* sc_c, int enable, cudaStream_t st) {
  jacobi_scale_cams_kernel<<<(D + 255) / 256, 256, 0, st>>>(D, hdiag, sc_c, enable);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_point_prep(int N, const double* H_pp, const double* g_p, const double* sc_p, const uint8_t* point_const,
                      double radius, double min_diag, double max_diag, double* M, double* q, double* dpp,
                      double* scal, cudaStream_t st) {
  point_prep_kernel<<<(N + 127) / 128, 128, 0, st>>>(N, H_pp, g_p, sc_p, point_const, radius, min_diag, max_diag, M, q,
                                                     dpp, scal);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_assemble_hc(int S, int dc, int ns, int KR, int Dpad, const double* camrec, const double* shared_in,
                       double* Sraw, double* rhs, double* hdiag, double* gvec, ptrdiff_t mc_off, cudaStream_t st) {
  assemble_hc_kernel<<<S + (ns > 0 ? 1 : 0), 64, 0, st>>>(S, dc, ns, KR, Dpad, camrec, shared_in, Sraw, rhs, hdiag, gvec,
                                                          mc_off);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_z_transpose(int D, int N, int Dpad, const double* W, const double* M, const double* q, double* Zt,
                       double* rhs, ptrdiff_t mc_off, cudaStream_t st, unsigned long long* amax) {
  const size_t pitch = (size_t)(D + (D & 1));
  dim3 grid((D + 127) / 128, (N + ZB_NT - 1) / ZB_NT);
  z_build_kernel<<<grid, 128, 0, st>>>(D, N, Dpad, pitch, W, M, q, Zt, rhs, mc_off, amax, g_band_dev.rb_range);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
// reduce-scatter destinations of the running multi-GPU solve (set per iteration by csrc/ba_solve.cu; world <= 1: off)
FabricDev g_fabric_dev = {0, 0, {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}};

int launch_scale_damp(int D, int Dpad, double* A, const double* rhs, const double* hdiag, const double* sc,
                      const uint8_t* pconst, double radius, double min_diag, double max_diag, double* bvec,
                      cudaStream_t st) {
  dim3 grid((D + 255) / 256, D);
  scale_damp_kernel<<<grid, 256, 0, st>>>(D, Dpad, A, rhs, hdiag, sc, pconst, radius, min_diag, max_diag, bvec);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_cam_step(int D, const double* dcs, size_t dcs_stride, const double* sc, const double* hdiag, const double* gvec,
                    const uint8_t* pconst, double radius, double min_diag, double max_diag, double* d_c, double* scal,
                    cudaStream_t st) {
  cam_step_kernel<<<(D + 255) / 256, 256, 0, st>>>(D, dcs, dcs_stride, sc, hdiag, gvec, pconst, radius, min_diag, max_diag, d_c, scal);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_backsub(int D, int N, const double* W, const double* d_c, double* wacc, cudaStream_t st) {
  const size_t pitch = (size_t)(D + (D & 1));
  backsub_kernel<<<(N + 7) / 8, 256, 0, st>>>(D, N, pitch, W, d_c, wacc, g_band_dev.kb_rows, g_band_dev.arrow_row);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_point_step(int N, const double* M, const double* g_p, const double* wacc, const double* sc_p,
                      const double* dpp, const double* X, double radius, double* Xc, double* scal, cudaStream_t st) {
  point_step_kernel<<<(N + 127) / 128, 128, 0, st>>>(N, M, g_p, wacc, sc_p, dpp, X, radius, Xc, scal);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_cam_update(int S, int dc, int ns, int model, const double* d_c, const double* poses, const double* intr,
                      double* poses_c, double* intr_c, cudaStream_t st) {
  cam_update_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, dc, ns, model, d_c, poses, intr, poses_c, intr_c);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_extract_gvec(int S, int dc, int ns, int KR, const double* camrec, const double* shared_in, double* gvec,
                        cudaStream_t st) {
  const int D = S * dc + ns;
  extract_gvec_kernel<<<(D + 255) / 256, 256, 0, st>>>(S, dc, ns, KR, camrec, shared_in, gvec);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}
int launch_gradmax(int D, int N, const double* gvec, const uint8_t* pconst, const double* g_p,
                   const uint8_t* point_const, double* scal, cudaStream_t st) {
  const int n = D > N * 3 ? D : N * 3;
  gradmax_kernel<<<(n + 255) / 256, 256, 0, st>>>(D, N, gvec, pconst, g_p, point_const, scal);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}

}  // namespace vgg
