// Blocked right-looking Cholesky of the reduced camera system (row-major, lower triangle, in place) -- the
// factorisation inside Ceres' DENSE_SCHUR (LAPACK potrf reached from pycolmap.bundle_adjustment), and the largest
// serial piece of a bundle-adjustment iteration: n = 2403 at 400 frames (bordered with the right-hand side), 4.6 GFLOP
// of float64 whose cost is a dependency chain, not arithmetic.  128-column panels; per panel
//   chol_panel_kernel   EVERY CTA re-factors the 128x128 diagonal block in shared memory (cta_chol128 below) with its
//                       own 16 panel rows riding along, so no CTA waits for another one and the rows come out solved;
//                       it writes them back together with their transpose (the upper triangle ends up holding L^T,
//                       which is what the backward substitution kernel, csrc/trsv.cu, streams row by row), then --
//                       fused schedule -- waits for the eight CTAs that own block row k+1, loads those 128 rows and
//                       applies this panel's update to its own rows of block column k+1 with DMMA + f64 REDs.  The
//                       next panel kernel follows on the same stream.  <= 143 CTAs: one wave.
//   chol_update_kernel  A22 -= P P^T on 64x64 tiles with mma.sync.m8n8k4.f64 (SASS DMMA) for block columns >= k+2, on a
//                       low-priority side stream; one K half of both operands in shared memory at a time (68 KB) so that
//                       its CTAs run NEXT TO the panel CTAs of the following step (152 KB) on the same SMs.
// The whole launch sequence is captured once per (matrix, order) into a CUDA graph.  Matrices of fewer than three
// panels (n <= 256) run in program order instead: update, then the next panel, all on the caller's stream.
// Measured slower on a B200 and removed (profiles/README.md): the first r02 schedule (a separate critical-path update
// kernel with the next panel on a side stream), a persistent trailing-update kernel (0.920 vs 0.890 ms at n = 2403) and
// the one-pivot-per-step 8x8 leaf.
#include <algorithm>
#include <map>
#include <vector>
#include <tuple>
#include "common.cuh"

namespace vgg {

constexpr int CB = 128;       // panel width
constexpr int CLD = 132;      // shared-memory row stride (doubles): rows 16-byte aligned, DMMA fragment loads conflict-free
constexpr int C_RPC = 16;     // panel rows per CTA in the triangular solve
constexpr int CT = 64;        // trailing-update tile
constexpr int C_THREADS = 256;

__device__ __forceinline__ void chol_dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// Cholesky of the 128x128 block in shared memory Ls (row stride CLD) by the whole CTA (256 threads).  Lower triangle
// in, L out (entries above the diagonal are left undefined).  dinv[j] = 1 / L[j][j].  Returns 0 or 1 + first bad pivot.
// Two levels (r02 profile of the one-level version: 77 us per panel, the 4x4-tile rank-8 updates of the whole
// trailing block ran into 8-way bank conflicts and 128 FMA instructions per 16 outputs):
//   * four 32-column sub-panels; inside one, 8-column micro-panels: (a) 8x8 leaf by warp 0 (one row per lane, pivot
//     columns through shuffles, two pivots per step), (b) one thread per row below solves its 8 entries against the
//     pre-scaled leaf, (c) rank-8 update of the REST OF THE SUB-PANEL only (<= 24 columns), two threads per row, by warps
//     1..7 WHILE warp 0 already prepares and factors the next leaf (the pivot chain is the critical path);
//   * after each sub-panel ONE rank-32 update of everything to its right with mma.sync.m8n8k4.f64 (DMMA), 32x16 warp
//     tiles straight from the row-major block (row stride 132: conflict-free fragments), tiles handed out through a
//     shared counter; warp 0 takes the tile with the next leaf first and factors it under the other warps' tiles.
// r02 one-CTA probe (tools/microbench.py chol128, cycles): 55.5 k with the first leaf -> 47.9 k (hardware f64 rsqrt seed,
// two-pivot leaf, per-lane look-ahead prep, overlapped sub-panel leaves); floor from the FP64 pipe alone: ~13 k.
// 1/sqrt(p) for normal p > 0: the hardware's double-precision seed (rsqrt.approx.ftz.f64 -> MUFU.RSQ64H, relative error
// 2^-22.4 over the whole double range) + two Newton steps (-> 2^-44 -> below one ulp).  No float round trip, no range
// check and no select in front of it: this sits on the 128-deep pivot chain of every panel, and the first version
// (float seed: F2F, FSETP, FMUL, MUFU, FMUL, F2F before the first Newton step, behind a DSETP/FSEL range guard) spent
// about as long getting to the seed as refining it.  Callers test the pivot in parallel and discard the result if the
// pivot was not a normal positive number.
__device__ __forceinline__ double fast_rsqrt(double p) {
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(p));
  const double hp = 0.5 * p;
  r = r * fma(-hp * r, r, 1.5);
  r = r * fma(-hp * r, r, 1.5);
  return r;
}
constexpr double CHOL_PMIN = 2.2250738585072014e-308;      // smallest normal double: pivots below it count as non-positive

// PROBE adds clock64 phase counters for tools/microbench.py chol128 (threads 0 and 32 = warp 0 / warp 1; prof[warp][phase], see the MARK sites).
//
// xr (0 or C_RPC) extra rows stored right below the block (rows 128 .. 128+xr-1 of Ls) ride along: they take part in the
// micro-panel solves and in the rank-8 / rank-32 updates, so when the block is factored they hold X = A_ik L^-T -- the
// panel rows this CTA owns -- with no separate triangular solve afterwards (r02: that solve was a 128-step
// multiply/shuffle/FMA chain, ~3 us after every POTRF128, plus a transposing pass over the block to feed it).
template <bool PROBE>
__device__ __forceinline__ int cta_chol128(double* Ls, double* dinv, int* fail_sm, int tid, int xr,
                                           long long* prof = nullptr) {
  const int lane = tid & 31, warp = tid >> 5;
  // Lh[m][k] = L[m][k] / L[m][m] (k < m) of the current 8 x 8 leaf: with the rows pre-scaled the solve of a row below it
  // is ONE fma per column on its dependency chain instead of a multiply and an fma (r02 probe: that phase was 12 % of
  // the POTRF128, all of it latency)
  __shared__ __align__(16) double Lh[64];
  if (tid == 0) *fail_sm = 0;
  __syncthreads();
  // packed lower-triangle entry of an 8 x 8 block owned by this lane in the look-ahead prep: e = lane (and lane + 32 for
  // lanes 0..3; the other lanes recompute entry 35 and drop it)
  auto tri_row = [](int e) { return (e >= 1) + (e >= 3) + (e >= 6) + (e >= 10) + (e >= 15) + (e >= 21) + (e >= 28); };
  const int pi0 = tri_row(lane), pj0 = lane - pi0 * (pi0 + 1) / 2;
  const int e1 = lane < 4 ? lane + 32 : 35;
  const int pi1 = tri_row(e1), pj1 = e1 - pi1 * (pi1 + 1) / 2;
  long long pacc[6] = {0, 0, 0, 0, 0, 0}, plast = 0;
  const bool ptid = PROBE && (tid == 0 || tid == 32);
  if (ptid) plast = clock64();
#define CHOL_MARK(ph)                         \
  if (ptid) {                                 \
    const long long t_ = clock64();           \
    pacc[ph] += t_ - plast;                   \
    plast = t_;                               \
  }
  // 8x8 leaf by warp 0: one row per lane (lanes 8..31 mirror lanes 0..7), pivot columns through shuffles, TWO pivots
  // per step.  For the 2x2 block [[A, B], [B, C]] both reciprocal square roots come from independent inputs:
  //   1/L00 = rsqrt(A),   1/L11 = rsqrt(C - B^2/A) = sqrt(A) * rsqrt(A C - B^2),
  // so the serial chain per PAIR is shuffle -> det -> rsqrt -> two scalings -> shuffle -> two FMAs (~220 cycles) where the
  // one-pivot-per-step version paid ~300 cycles per pivot (r02 source-correlated profile: 45 % of the panel kernel's
  // warp samples waited on barriers behind this chain).  det = A C - B^2 carries the same relative error bound as
  // C - (B/sqrt A)^2 (both ~ eps C / (C - B^2/A)); if A C leaves the comfortable exponent range the second pivot falls
  // back to the sequential formula (warp-uniform branch).  A shuffle-free variant (every lane holds the whole
  // 36-element triangle) measured SLOWER: panel 51.6 vs 48.6 us -- 36 broadcast loads + 64 predicated stores per leaf
  // cost more than the shuffles they replace.
  auto leaf = [&](int c0) {
    double a[8];
    const int r = c0 + (lane & 7);
#pragma unroll
    for (int c = 0; c < 8; c += 2) {
      const double2 v = *reinterpret_cast<const double2*>(Ls + r * CLD + c0 + c);
      a[c] = v.x;
      a[c + 1] = v.y;
    }
    int fail = 0;
    double mydinv = 1.0;
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const double A = __shfl_sync(0xffffffffu, a[j], j);
      const double B = __shfl_sync(0xffffffffu, a[j], j + 1);
      const double C = __shfl_sync(0xffffffffu, a[j + 1], j + 1);
      const double AC = A * C;
      const double det = fma(-B, B, AC);
      double ia = fast_rsqrt(A);
      double ib = (A * ia) * fast_rsqrt(det);
      double l10 = B * ia;
      // the tests run in the shadow of the two rsqrt chains; the branch is warp-uniform (every lane holds A, B, C)
      const bool good = A >= CHOL_PMIN && det >= CHOL_PMIN && AC < 1e280 && AC > 1e-280;
      if (!good) {
        if (!(A >= CHOL_PMIN)) {
          if (fail == 0) fail = c0 + j + 1;
          ia = 1.0;
          l10 = B;
        }
        const double p1 = fma(-l10, l10, C);
        if (!(p1 >= CHOL_PMIN)) {
          if (fail == 0) fail = c0 + j + 2;
          ib = 1.0;
        } else {
          ib = rsqrt(p1);
        }
      }
      const double x0 = a[j] * ia;                          // lane j: A * ia = sqrt(A)
      const double x1 = fma(-x0, l10, a[j + 1]) * ib;       // lane j+1: (C - l10^2) / sqrt(C - l10^2)
      a[j] = x0;
      a[j + 1] = x1;
      if (lane == j) {
        dinv[c0 + j] = ia;
        dinv[c0 + j + 1] = ib;
        mydinv = ia;
      }
      if (lane == j + 1) mydinv = ib;
#pragma unroll
      for (int c = j + 2; c < 8; ++c) {
        const double l0 = __shfl_sync(0xffffffffu, x0, c);
        const double l1 = __shfl_sync(0xffffffffu, x1, c);
        if (lane >= c) a[c] = fma(-x1, l1, fma(-x0, l0, a[c]));
      }
    }
    if (lane < 8) {
#pragma unroll
      for (int c = 0; c < 8; ++c) Ls[r * CLD + c0 + c] = (c <= lane) ? a[c] : 0.0;
#pragma unroll
      for (int c = 0; c < 8; ++c) Lh[lane * 8 + c] = (c < lane) ? a[c] * mydinv : 0.0;
    }
    if (lane == 0 && fail && *fail_sm == 0) *fail_sm = fail;
  };
  // C[r][j] -= sum_k L[r][c0+k] L[j][c0+k] for j = jb, jb+js, ... <= jend (two columns in flight)
  auto row_update = [&](int r, int c0, int jb, int js, int jend) {
    double li[8];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
      const double2 v = *reinterpret_cast<const double2*>(Ls + r * CLD + c0 + k);
      li[k] = v.x;
      li[k + 1] = v.y;
    }
    int j = jb;
    for (; j + js <= jend; j += 2 * js) {
      const double* l0 = Ls + j * CLD + c0;
      const double* l1 = Ls + (j + js) * CLD + c0;
      double s0 = Ls[r * CLD + j], s1 = Ls[r * CLD + j + js];
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        const double2 u = *reinterpret_cast<const double2*>(l0 + k);
        const double2 w = *reinterpret_cast<const double2*>(l1 + k);
        s0 = fma(-li[k], u.x, s0);
        s1 = fma(-li[k], w.x, s1);
        s0 = fma(-li[k + 1], u.y, s0);
        s1 = fma(-li[k + 1], w.y, s1);
      }
      Ls[r * CLD + j] = s0;
      Ls[r * CLD + j + js] = s1;
    }
    if (j <= jend) {
      const double* l0 = Ls + j * CLD + c0;
      double s0 = Ls[r * CLD + j];
#pragma unroll
      for (int k = 0; k < 8; k += 2) {
        const double2 u = *reinterpret_cast<const double2*>(l0 + k);
        s0 = fma(-li[k], u.x, s0);
        s0 = fma(-li[k + 1], u.y, s0);
      }
      Ls[r * CLD + j] = s0;
    }
  };
  if (warp == 0) leaf(0);
  __syncthreads();
  CHOL_MARK(0)
  for (int sp = 0; sp < CB / 32; ++sp) {
    const int c32 = sp * 32;
    for (int mp = 0; mp < 4; ++mp) {
      const int c0 = c32 + mp * 8;
      // (b) rows below the micro-block: x L^T = a, one thread per row
      {
        const int r = c0 + 8 + tid;
        if (r < CB + xr) {
          double x[8];
#pragma unroll
          for (int c = 0; c < 8; c += 2) {
            const double2 v = *reinterpret_cast<const double2*>(Ls + r * CLD + c0 + c);
            x[c] = v.x;
            x[c + 1] = v.y;
          }
#pragma unroll
          for (int m = 0; m < 8; ++m) x[m] *= dinv[c0 + m];            // all eight in parallel
#pragma unroll
          for (int m = 1; m < 8; ++m) {
#pragma unroll
            for (int k = 0; k < m; ++k) x[m] = fma(-x[k], Lh[m * 8 + k], x[m]);      // only k = m-1 waits for the chain
          }
#pragma unroll
          for (int c = 0; c < 8; c += 2) *reinterpret_cast<double2*>(Ls + r * CLD + c0 + c) = make_double2(x[c], x[c + 1]);
        }
      }
      __syncthreads();
      CHOL_MARK(1)
      // (c) rank-8 update of the remaining columns of THIS sub-panel (c0+8 .. c32+31), all rows below -- with one
      //     micro-panel of lookahead: warp 0 first finishes the next 8x8 diagonal block and factors it (the pivot chain,
      //     ~1.3k cycles) while warps 1..7 update everything else (two threads per row, alternate columns)
      if (mp < 3) {
        const int n0 = c0 + 8;                                   // first row/column of the next micro-panel
        if (warp == 0) {
          // the next leaf's lower triangle, one entry (i, j) per lane (36 entries: lanes 0..3 take a second one): a
          // length-8 dot product in two chains.  (r02 probe: eight lanes walking their rows cost ~900 of the ~2300
          // cycles this section took per micro-panel -- and the section is the critical path of the factorisation.)
          {
            const double* ri = Ls + (n0 + pi0) * CLD + c0;
            const double* rj = Ls + (n0 + pj0) * CLD + c0;
            const double* ri1 = Ls + (n0 + pi1) * CLD + c0;
            const double* rj1 = Ls + (n0 + pj1) * CLD + c0;
            double s0 = Ls[(n0 + pi0) * CLD + n0 + pj0], s1 = 0.0;
            double u0 = Ls[(n0 + pi1) * CLD + n0 + pj1], u1 = 0.0;
#pragma unroll
            for (int k = 0; k < 8; k += 4) {
              const double2 a0 = *reinterpret_cast<const double2*>(ri + k), a1 = *reinterpret_cast<const double2*>(ri + k + 2);
              const double2 b0 = *reinterpret_cast<const double2*>(rj + k), b1 = *reinterpret_cast<const double2*>(rj + k + 2);
              const double2 c0v = *reinterpret_cast<const double2*>(ri1 + k), c1v = *reinterpret_cast<const double2*>(ri1 + k + 2);
              const double2 d0 = *reinterpret_cast<const double2*>(rj1 + k), d1 = *reinterpret_cast<const double2*>(rj1 + k + 2);
              s0 = fma(-a0.x, b0.x, s0);
              s1 = fma(-a0.y, b0.y, s1);
              u0 = fma(-c0v.x, d0.x, u0);
              u1 = fma(-c0v.y, d0.y, u1);
              s0 = fma(-a1.x, b1.x, s0);
              s1 = fma(-a1.y, b1.y, s1);
              u0 = fma(-c1v.x, d1.x, u0);
              u1 = fma(-c1v.y, d1.y, u1);
            }
            Ls[(n0 + pi0) * CLD + n0 + pj0] = s0 + s1;
            if (lane < 4) Ls[(n0 + pi1) * CLD + n0 + pj1] = u0 + u1;
          }
          __syncwarp();
          leaf(n0);
        } else {
          const int t = tid - 32;                                 // 224 threads: row = n0 + t/2 (skipping nothing), half
          for (int rr = t >> 1; n0 + rr < CB + xr; rr += 112) {
            const int r = n0 + rr, half = t & 1;
            const int jend = min(r, c32 + 31);
            // rows of the next leaf block (r < n0+8) own only columns right of it?  no: their columns <= r all lie inside
            // the leaf block, which warp 0 handles; other rows skip nothing
            if (r < n0 + 8) continue;
            row_update(r, c0, n0 + half, 2, jend);
          }
        }
        CHOL_MARK(2)
        __syncthreads();
        CHOL_MARK(3)
      }
    }
    // rank-32 update of the block to the right of the sub-panel: C[i][j] -= sum_k L[i][c32+k] L[j][c32+k], i >= j >= c32+32
    const int t0 = c32 + 32;
    const int nrb = (CB - t0) / 32;                  // 32-row blocks: 3, 2, 1, 0
    if (nrb > 0) {
      const int ntile = nrb * (nrb + 1);             // sum over rb of (2 rb + 2) 16-column tiles
      const int nxt = xr ? (CB - t0) / 16 : 0;       // 16 x 16 tiles of the ride-along rows (two 8-row MMA blocks)
      const int g = lane >> 2, q = lane & 3;
      // warp 0 updates tile 0 (it holds the next sub-panel's first 8 x 8 block), then factors that block while warps
      // 1..7 work through the remaining tiles round-robin (r02 probe: the three unoverlapped leaves were 9 % of the
      // POTRF128).  Handing the tiles out through a shared counter instead was SLOWER (phase 14.0 k -> 18.2 k cycles):
      // warp 0 then picks up a late tile after its leaf and becomes the straggler of the phase.
      bool leaf_pending = warp == 0;
      for (int t = warp == 0 ? 0 : warp; t < ntile + nxt; t += (warp == 0 ? ntile + nxt : C_THREADS / 32 - 1)) {
        int R0, C0, nrow8 = 4;
        if (t < ntile) {
          int rb = 0, cb = t;
          while (cb >= 2 * rb + 2) { cb -= 2 * rb + 2; ++rb; }
          R0 = t0 + rb * 32;
          C0 = t0 + cb * 16;
        } else {
          R0 = CB;
          C0 = t0 + (t - ntile) * 16;
          nrow8 = 2;
        }
        double c[4][2][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) c[i][j][0] = c[i][j][1] = 0.0;
        const double* arow = Ls + (R0 + g) * CLD + c32 + q;
        const double* brow = Ls + (C0 + g) * CLD + c32 + q;
#pragma unroll
        for (int k4 = 0; k4 < 8; ++k4) {
          double a[4], b[2];
#pragma unroll
          for (int i = 0; i < 4; ++i) a[i] = (i < nrow8) ? arow[i * 8 * CLD + k4 * 4] : 0.0;
#pragma unroll
          for (int j = 0; j < 2; ++j) b[j] = brow[j * 8 * CLD + k4 * 4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (i < nrow8) {                               // warp-uniform
#pragma unroll
              for (int j = 0; j < 2; ++j) chol_dmma(c[i][j][0], c[i][j][1], a[i], b[j]);
            }
          }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (i >= nrow8) continue;
          const int r = R0 + i * 8 + g;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int col = C0 + j * 8 + 2 * q;
            if (col > r) continue;
            double* pp = Ls + r * CLD + col;
            if (col + 1 <= r) {
              double2 v = *reinterpret_cast<double2*>(pp);
              v.x -= c[i][j][0];
              v.y -= c[i][j][1];
              *reinterpret_cast<double2*>(pp) = v;
            } else {
              *pp -= c[i][j][0];
            }
          }
        }
        if (leaf_pending) {
          __syncwarp();
          leaf(t0);
          leaf_pending = false;
        }
      }
      CHOL_MARK(4)
      __syncthreads();
      CHOL_MARK(5)
    }
  }
#undef CHOL_MARK
  if (ptid) {
#pragma unroll
    for (int i = 0; i < 6; ++i) prof[(tid == 32 ? 6 : 0) + i] = pacc[i];
  }
  return *fail_sm;
}

// one-CTA probe: factor a 128 x 128 block `reps` times (reloading it each time), report the cycles of the last pass
__global__ void __launch_bounds__(C_THREADS, 1) chol128_probe_kernel(const double* __restrict__ A, double* __restrict__ L,
                                                                      long long* __restrict__ prof, int reps, int xr) {
  extern __shared__ __align__(16) double cp_smem[];
  __shared__ double dinv[CB];
  __shared__ int fail_sm;
  const int tid = threadIdx.x;
  long long total = 0;
  for (int rep = 0; rep < reps; ++rep) {
    for (int e = tid; e < CB * CB; e += C_THREADS) cp_smem[(e >> 7) * CLD + (e & 127)] = A[e];
    for (int e = tid; e < xr * CB; e += C_THREADS)          // ride-along rows: copies of the block's last rows
      cp_smem[(CB + (e >> 7)) * CLD + (e & 127)] = A[(CB - xr + (e >> 7)) * CB + (e & 127)];
    __syncthreads();
    const long long t0 = clock64();
    cta_chol128<true>(cp_smem, dinv, &fail_sm, tid, xr, prof);
    __syncthreads();
    total = clock64() - t0;
  }
  if (tid == 0) prof[12] = total;
  for (int e = tid; e < CB * CB; e += C_THREADS) L[e] = ((e & 127) <= (e >> 7)) ? cp_smem[(e >> 7) * CLD + (e & 127)] : 0.0;
}

// grid.x = 1 + number of 16-row chunks below the diagonal block; block 256.  Every CTA factors the diagonal block
// redundantly with its own 16 panel rows riding along (xr = C_RPC), so those rows come out solved.  CTA 0 stores the
// factored block: L^T into the strict upper triangle in place (nobody reads it), L itself into the side buffer Ldiag --
// the other CTAs of this launch may still be loading the unfactored block; CTA 0 of the NEXT panel's launch moves it
// into place (the last panel, a single CTA, writes its block directly).
//
// fuse != 0: the CTA then applies THIS panel's update to its own rows of the NEXT block column,
//   A[r0.., t0..t0+127] -= X P^T,   X = its solved rows,  P = L[t0..t0+127][k0..k0+127]  (block row k+1 of the panel),
// so that column is complete when the kernel ends and the next panel kernel can follow directly (r02: the separate
// critical-path update kernel and its two cross-stream graph edges cost ~12 us per panel step on top of the ~9 us the
// kernel ran).  P is produced by CTAs 1..8 of this launch: they publish their rows (fence + flags[panel]++), everyone
// spins on the counter (bounded), then loads P through L2.  A CTA only ever waits for lower-numbered CTAs, which the
// hardware dispatched before it, so the wait cannot deadlock even when the grid is not co-resident.  The subtraction
// uses f64 REDs: the trailing-update kernel of the PREVIOUS panel may still be adding into the same tiles.
constexpr int CHOL_SPIN_LIMIT = 1 << 22;
constexpr int CHOL_INFO_STALLED = 0x7fffffff;

__global__ void __launch_bounds__(C_THREADS, 1) chol_panel_kernel(int n, int lda, int k0, double* __restrict__ A,
                                                                   double* __restrict__ Ldiag /*[nblk][128*128]*/,
                                                                   int* __restrict__ info, int* __restrict__ flags,
                                                                   int fuse, int band_end, int arrow_lo) {
  // Rows below the diagonal block that can be non-zero in this block column: [k0+128, band_end) and [arrow_lo, n)
  // (band_end = arrow_lo = n: everything, the dense case).  The CTAs cover exactly these rows, 16 each.
  extern __shared__ __align__(16) double cp_smem[];
  double* Ls = cp_smem;                        // [128][CLD]
  double* Ts = cp_smem + CB * CLD;             // [16][CLD]: rows 128.. of the same array (ride-along rows)
  __shared__ double dinv[CB];
  __shared__ int fail_sm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = min(CB, n - k0);
  const bool solver = blockIdx.x > 0;
  const int chunks1r = (max(0, min(band_end, n) - (k0 + CB)) + C_RPC - 1) / C_RPC;   // banded: band_end is a multiple of 128
  const int cidx = (int)blockIdx.x - 1;
  const int r0 = cidx < chunks1r ? k0 + CB + cidx * C_RPC : arrow_lo + (cidx - chunks1r) * C_RPC;
  // diagonal block (rows < nb: whole 128-double rows, the part above the diagonal is never read; identity padding
  // beyond nb) and this CTA's 16 panel rows: cp.async, all 16-byte chunks in flight at once (r02: the plain
  // load -> store loop serialised 32 L2 round trips per thread, a third of the kernel)
  for (int e = tid; e < CB * (CB / 2); e += C_THREADS) {
    const int i = e >> 6, j = (e & 63) * 2;
    if (i < nb) {
      cp_async16(Ls + i * CLD + j, A + (size_t)(k0 + i) * lda + k0 + j);
    } else {
      *reinterpret_cast<double2*>(Ls + i * CLD + j) = make_double2(j == i ? 1.0 : 0.0, j + 1 == i ? 1.0 : 0.0);
    }
  }
  for (int e = tid; e < C_RPC * (CB / 2); e += C_THREADS) {
    const int r = e >> 6, j = (e & 63) * 2;
    if (solver && r0 + r < n) cp_async16(Ts + r * CLD + j, A + (size_t)(r0 + r) * lda + k0 + j);
    else *reinterpret_cast<double2*>(Ts + r * CLD + j) = make_double2(0.0, 0.0);
  }
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  const int fail = cta_chol128<false>(Ls, dinv, &fail_sm, tid, C_RPC);
  if (fail && blockIdx.x == 0 && tid == 0) atomicCAS(info, 0, k0 + fail);
  if (!solver) {
    // the last panel has no other CTA that could still be loading the block: its factor goes straight into place
    const bool alone = gridDim.x == 1;
    double* dst = Ldiag + (size_t)(k0 / CB) * CB * CB;
    for (int e = tid; e < CB * CB; e += C_THREADS) {
      const int i = e >> 7, j = e & 127;
      if (i < nb && j < nb) {
        if (j > i) A[(size_t)(k0 + i) * lda + k0 + j] = Ls[j * CLD + i];      // L^T (transposed read: CTA 0 is off the critical path)
        else if (alone) A[(size_t)(k0 + i) * lda + k0 + j] = Ls[i * CLD + j];
        else dst[e] = Ls[i * CLD + j];
      }
    }
    // ... and the PREVIOUS panel's parked factor moves into place now (its launch is over, nobody reads that block again)
    if (k0 > 0) {
      const double* src = Ldiag + (size_t)(k0 / CB - 1) * CB * CB;
      double* blk = A + (size_t)(k0 - CB) * lda + (k0 - CB);
      // eight loads in flight per thread (r02: the plain load -> store loop ran one L2 round trip per element and made
      // CTA 0 the last CTA of every panel launch: 0.90 -> 1.05 ms)
      for (int e0 = tid; e0 < CB * CB; e0 += 8 * C_THREADS) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = e0 + u * C_THREADS;
          v[u] = ((e & 127) <= (e >> 7)) ? __ldcg(src + e) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int e = e0 + u * C_THREADS;
          const int i = e >> 7, j = e & 127;
          if (j <= i) blk[(size_t)i * lda + j] = v[u];
        }
      }
    }
    return;
  }
  // row-major store of the solved rows ...
  for (int e = tid; e < C_RPC * CB; e += C_THREADS) {
    const int r = e >> 7, c = e & 127;
    if (r0 + r < n && c < nb) A[(size_t)(r0 + r) * lda + k0 + c] = Ts[r * CLD + c];
  }
  // ... and their transpose into the upper triangle (16 consecutive doubles = one 128-byte segment per column c)
  for (int e = tid; e < C_RPC * CB; e += C_THREADS) {
    const int c = e >> 4, r = e & 15;
    if (r0 + r < n && c < nb) A[(size_t)(k0 + c) * lda + r0 + r] = Ts[r * CLD + c];
  }
  if (!fuse) return;

  // ---- fused update of block column k+1 with this panel
  const int t0 = k0 + CB;
  // CTAs 1..nprod own block row k+1 (the band's first block, or the arrow block when it is the next one); a block
  // row that is structurally zero in this column has no producers and there is nothing to subtract
  const bool p_active = band_end > t0 || arrow_lo == t0;
  const int nprod = p_active ? min(CB / C_RPC, (int)gridDim.x - 1) : 0;
  if (nprod == 0) return;
  int* flag = flags + k0 / CB;
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    if ((int)blockIdx.x <= nprod) atomicAdd(flag, 1);           // after the fence: this CTA's rows are visible device-wide
    int spins = 0, seen;
    do {
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(seen) : "l"(flag) : "memory");
    } while (seen < nprod && ++spins < CHOL_SPIN_LIMIT);
    if (seen < nprod) atomicCAS(info, 0, CHOL_INFO_STALLED);
  }
  __syncthreads();
  // P = rows t0 .. t0+127 of the panel -> Ls (the factored block is no longer needed here); two K halves
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    for (int e = tid; e < CB * 16; e += C_THREADS) {
      const int row = e >> 4, ch = (e & 15) * 4 + half * 64;
      double* dst = Ls + row * CLD + ch;
      if (t0 + row < n) {
        const double* src = A + (size_t)(t0 + row) * lda + k0 + ch;
        cp_async16(dst, src);
        cp_async16(dst + 2, src + 2);
      } else {
        *reinterpret_cast<double2*>(dst) = make_double2(0.0, 0.0);
        *reinterpret_cast<double2*>(dst + 2) = make_double2(0.0, 0.0);
      }
    }
    cp_async_commit();
  }
  {
    const int g = lane >> 2, q = lane & 3;
    double c[2][2][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) c[i][j][0] = c[i][j][1] = 0.0;
    const double* arow = Ts + g * CLD + q;
    const double* brow = Ls + (warp * 16 + g) * CLD + q;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      if (half == 0) cp_async_wait<1>();
      else cp_async_wait<0>();
      __syncthreads();
#pragma unroll 4
      for (int k4 = half * 16; k4 < half * 16 + 16; ++k4) {
        double a[2], b[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) a[i] = arow[i * 8 * CLD + k4 * 4];
#pragma unroll
        for (int j = 0; j < 2; ++j) b[j] = brow[j * 8 * CLD + k4 * 4];
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) chol_dmma(c[i][j][0], c[i][j][1], a[i], b[j]);
      }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int r = r0 + i * 8 + g;
      if (r >= n) continue;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const int col = t0 + warp * 16 + j * 8 + 2 * q;
        double* p = A + (size_t)r * lda + col;
        if (col <= r) atomicAdd(p, -c[i][j][0]);
        if (col + 1 <= r) atomicAdd(p + 1, -c[i][j][1]);
      }
    }
  }
}

// A[t0.., t0..] -= P P^T (lower part), P = A[t0.., k0..k0+127].  64x64 tiles (bi, bj), bj <= bi, one per CTA, 8 warps
// as 2x4, warp tile 32x16.  mode 0 = all tile columns; mode 4 = tile columns 2 and 3 only (block column k+2, which the
// fused panel kernel of the next step is adding into at the same time: f64 REDs), mode 5 = tile columns >= 4 (REDs on 4
// and 5): the two pieces of the trailing update with different deadlines.
// Shared memory holds ONE K half (64 panel columns) of both operands at a time, row stride 68 doubles (fragment loads
// conflict-free like stride 132): 68 KB per CTA instead of 135 KB, so an update CTA fits on an SM NEXT TO a panel CTA
// (152 KB) and two or three fit on a free SM.  r02 launch list of the previous version (whole K resident, one CTA per
// SM): the panel kernel's <= 143 latency-bound CTAs held their SMs for the whole step and the trailing update ran
// after them, not beside them -- the factorisation took the SUM of all its kernels (0.90 ms).
constexpr int CUD = 68;
__global__ void __launch_bounds__(C_THREADS, 2) chol_update_kernel(int n, int lda, int k0, int t0, int mode,
                                                                    double* __restrict__ A, int band_end, int arrow_lo,
                                                                    int all_red) {
  constexpr int TM = 64;                          // tile rows
  constexpr int WN = 4;                           // warps along the 64 tile columns
  constexpr int NJ = 64 / WN / 8;                 // 8-column MMA tiles per warp
  extern __shared__ __align__(16) double cu_smem[];
  double* As = cu_smem;                         // [TM][CUD]
  double* Bs = cu_smem + TM * CUD;              // [64][CUD]
  int bi, bj;
  {
    const int t = blockIdx.x;
    if (mode == 4) {                         // tile columns 2 and 3 only (= block column k+2)
      const int T = (max(0, min(band_end, n) - t0) + 63) / 64 + (band_end >= n ? 0 : (n - arrow_lo + 63) / 64);
      if (t < T - 2) { bi = 2 + t; bj = 2; }
      else { bi = 3 + (t - (T - 2)); bj = 3; }
    } else {
      bi = (int)((sqrtf(8.0f * (float)t + 1.0f) - 1.0f) * 0.5f);
      while ((bi + 1) * (bi + 2) / 2 <= t) ++bi;
      while (bi * (bi + 1) / 2 > t) --bi;
      bj = t - bi * (bi + 1) / 2;
      const int skip = mode == 5 ? 4 : 0;
      bi += skip;
      bj += skip;
    }
  }
  const bool diag = bi == bj;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // banded matrices: 64-row tile v of the ACTIVE rows -- the band part [t0, band_end) first, then the arrow part
  // [arrow_lo, n) (band_end = n: the plain dense mapping)
  const int T1v = band_end >= n ? (1 << 30) : (band_end - t0) / 64;
  auto vrow = [&](int v) { return v < T1v ? t0 + v * 64 : arrow_lo + (v - T1v) * 64; };
  const int ri = vrow(bi), rj = vrow(bj);
  const double* bs = diag ? As : Bs;
  const int wm = warp / WN, wn = warp % WN;
  const int g = lane >> 2, q = lane & 3;
  double c[4][NJ][2];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < NJ; ++j) c[i][j][0] = c[i][j][1] = 0.0;
  const double* arow = As + (wm * 32 + g) * CUD + q;
  const double* brow = bs + (wn * (8 * NJ) + g) * CUD + q;
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    if (half) __syncthreads();                      // everyone is done with the first half's fragments
    // panel rows, row-major (k contiguous)
    for (int e = tid; e < (TM + 64) * 16; e += C_THREADS) {
      const int row = e >> 4, ch = (e & 15) * 4;     // 4 doubles (two 16-byte chunks) per thread-step
      const bool isA = row < TM;
      if (!isA && diag) continue;
      const int grow = isA ? ri + row : rj + (row - TM);
      double* dst = (isA ? As + row * CUD : Bs + (row - TM) * CUD) + ch;
      if (grow < n) {
        const double* src = A + (size_t)grow * lda + k0 + half * 64 + ch;
        cp_async16(dst, src);
        cp_async16(dst + 2, src + 2);
      } else {
        *reinterpret_cast<double2*>(dst) = make_double2(0.0, 0.0);
        *reinterpret_cast<double2*>(dst + 2) = make_double2(0.0, 0.0);
      }
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
#pragma unroll 4
    for (int k4 = 0; k4 < 16; ++k4) {
      double a[4], b[NJ];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = arow[i * 8 * CUD + k4 * 4];
#pragma unroll
      for (int j = 0; j < NJ; ++j) b[j] = brow[j * 8 * CUD + k4 * 4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) chol_dmma(c[i][j][0], c[i][j][1], a[i], b[j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = ri + wm * 32 + i * 8 + g;
    if (r >= n) continue;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int col = rj + wn * (8 * NJ) + j * 8 + 2 * q;
      if (col > r) continue;                         // lower triangle only (col <= r < n)
      double* p = A + (size_t)r * lda + col;
      if (all_red || mode == 4 || (mode == 5 && bj < 6)) {
        atomicAdd(p, -c[i][j][0]);
        if (col + 1 <= r) atomicAdd(p + 1, -c[i][j][1]);
      } else if (col + 1 <= r) {
        double2 v = *reinterpret_cast<double2*>(p);
        v.x -= c[i][j][0];
        v.y -= c[i][j][1];
        *reinterpret_cast<double2*>(p) = v;
      } else {
        *p -= c[i][j][0];
      }
    }
  }
}


size_t chol_workspace_doubles(int n) {
  const int nblk = (n + CB - 1) / CB;
  // factored diagonal blocks, parked until the end of the factorisation + one int per panel (the fused update's
  // "block row published" counters)
  return (size_t)nblk * CB * CB + (size_t)(nblk + 1) / 2 + 1;
}

namespace {

struct CholStreams {
  cudaStream_t side_lo = nullptr, side_mid = nullptr, cap = nullptr;
  cudaEvent_t ev_col = nullptr, ev_upd[2] = {nullptr, nullptr}, ev_bulk[3] = {nullptr, nullptr, nullptr};
  bool ready = false;
};

int chol_streams(CholStreams** out) {
  static thread_local CholStreams s;
  if (!s.ready) {
    int lo = 0, hi = 0;
    VGG_CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    // lo = least, hi = greatest priority.  The critical chain (panel steps) is captured on `cap` at the greatest
    // priority; the fused schedule's bulk updates go to side_lo at the least, so that a panel CTA is placed as soon as
    // an SM has room for it instead of queueing behind the remaining update CTAs.
    VGG_CUDA_CHECK(cudaStreamCreateWithPriority(&s.side_lo, cudaStreamNonBlocking, lo));
    VGG_CUDA_CHECK(cudaStreamCreateWithPriority(&s.side_mid, cudaStreamNonBlocking, (lo + hi) / 2));
    VGG_CUDA_CHECK(cudaStreamCreateWithPriority(&s.cap, cudaStreamNonBlocking, hi));
    VGG_CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_col, cudaEventDisableTiming));
    VGG_CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_upd[0], cudaEventDisableTiming));
    VGG_CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_upd[1], cudaEventDisableTiming));
    for (int i = 0; i < 3; ++i) VGG_CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_bulk[i], cudaEventDisableTiming));
    s.ready = true;
  }
  *out = &s;
  return VGG_OK;
}

int chol_set_attrs() {
  static bool done = false;
  if (done) return VGG_OK;
  VGG_CUDA_CHECK(cudaFuncSetAttribute(chol_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(sizeof(double) * (CB + C_RPC) * CLD)));
  VGG_CUDA_CHECK(cudaFuncSetAttribute(chol_update_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(sizeof(double) * 2 * CT * CUD)));
  done = true;
  return VGG_OK;
}

}  // namespace

// Block structure of a banded + arrow matrix (sequential / video problems; set by csrc/ba_solve.cu for the duration of
// a solve, empty = dense): in block column b the rows that can be non-zero below the diagonal block are the band
// [128 (b+1), 128 end_blk[b]) and the arrow [128 arrow_blk, n).  end_blk is non-decreasing (the envelope the
// factorisation fills) and end_blk[b] >= b + 2 while b + 1 < arrow_blk, so block row b+1 is always in the band.
std::vector<int> g_chol_band_end;
int g_chol_arrow_blk = 0;

namespace {

// The launch sequence on st and the side streams.
//   fused (nblk >= 3): step(b) = panel b + its update of block column b+1, all on st back to back; the rest of panel b's
//     trailing update (block columns >= b+2) runs on the side streams behind step(b) and has to be finished before
//     step(b+2) -- it shares block column b+2 with step(b+1)'s fused update, both sides use REDs there.
//   program order (nblk < 3): update(b) then panel(b+1), everything on st; the matrix is treated as dense.
int chol_enqueue(int n, int lda, double* A, double* Ldiag, int* info, int* flags, cudaStream_t st, CholStreams* cs) {
  const int nblk = (n + CB - 1) / CB;
  const size_t smem_p = sizeof(double) * (CB + C_RPC) * CLD;
  const size_t smem_u = sizeof(double) * 2 * CT * CUD;
  const bool fuse = nblk >= 3;
  const bool banded = fuse && (int)g_chol_band_end.size() >= nblk && g_chol_arrow_blk > 0;
  auto band_rows = [&](int b, int* band_end, int* arrow_lo) {
    if (!banded) {
      *band_end = *arrow_lo = n;
      return;
    }
    *band_end = std::min(n, g_chol_band_end[b] * CB);
    *arrow_lo = std::min(n, std::max(g_chol_arrow_blk * CB, *band_end));
    if (*band_end >= n || *arrow_lo <= *band_end) *band_end = *arrow_lo = n;      // no gap left: plain dense rows
  };
  auto panel = [&](int b) -> int {
    const int k0 = b * CB;
    int band_end, arrow_lo;
    band_rows(b, &band_end, &arrow_lo);
    const int below1 = std::max(0, std::min(band_end, n) - (k0 + CB));
    const int below2 = band_end >= n ? 0 : n - arrow_lo;
    const int chunks = (below1 + C_RPC - 1) / C_RPC + (below2 + C_RPC - 1) / C_RPC;
    chol_panel_kernel<<<1 + chunks, C_THREADS, smem_p, st>>>(n, lda, k0, A, Ldiag, info, flags, fuse ? 1 : 0, band_end, arrow_lo);
    VGG_LAUNCH_CHECK();
    return VGG_OK;
  };
  int rc;
  if ((rc = panel(0))) return rc;
  if (fuse) {
    // Panel b's trailing update in two pieces with different deadlines: U1(b) = block column b+2 (needed by step(b+2),
    // one step of slack, medium priority) and U2(b) = block columns >= b+3 (needed by step(b+3), two steps of slack,
    // lowest priority).  r02: as ONE kernel with one step of slack the update of the first six panels did not fit
    // next to the following step and 0.15 ms of it showed up on the critical path.
    bool have_u1[2] = {false, false}, have_u2[3] = {false, false, false};
    for (int b = 0; b + 1 < nblk; ++b) {
      const int k0 = b * CB, t0 = k0 + CB;
      int band_end, arrow_lo;
      band_rows(b, &band_end, &arrow_lo);
      const int T = (std::max(0, std::min(band_end, n) - t0) + CT - 1) / CT + (band_end >= n ? 0 : (n - arrow_lo + CT - 1) / CT);
      const int all_red = band_end >= n ? 0 : 1;     // banded: tile columns no longer map to consecutive block columns
      const int n_u1 = T > 2 ? (T - 2) + (T > 3 ? T - 3 : 0) : 0;
      const int n_u2 = T > 4 ? (T - 4) * (T - 3) / 2 : 0;
      have_u1[b & 1] = false;
      have_u2[b % 3] = false;
      if (n_u1 > 0) {
        VGG_CUDA_CHECK(cudaEventRecord(cs->ev_col, st));                 // step(b) done
        VGG_CUDA_CHECK(cudaStreamWaitEvent(cs->side_mid, cs->ev_col, 0));
        // U2(b-2) still writes block column b+2 with plain read-modify-writes (only its first block column uses REDs)
        if (b >= 2 && have_u2[(b - 2) % 3]) VGG_CUDA_CHECK(cudaStreamWaitEvent(cs->side_mid, cs->ev_bulk[(b - 2) % 3], 0));
        chol_update_kernel<<<n_u1, C_THREADS, smem_u, cs->side_mid>>>(n, lda, k0, t0, 4, A, band_end, arrow_lo, all_red);
        VGG_LAUNCH_CHECK();
        VGG_CUDA_CHECK(cudaEventRecord(cs->ev_upd[b & 1], cs->side_mid));
        have_u1[b & 1] = true;
        if (n_u2 > 0) {
          VGG_CUDA_CHECK(cudaStreamWaitEvent(cs->side_lo, cs->ev_col, 0));
          chol_update_kernel<<<n_u2, C_THREADS, smem_u, cs->side_lo>>>(n, lda, k0, t0, 5, A, band_end, arrow_lo, all_red);
          VGG_LAUNCH_CHECK();
          VGG_CUDA_CHECK(cudaEventRecord(cs->ev_bulk[b % 3], cs->side_lo));
          have_u2[b % 3] = true;
        }
      }
      // step(b+1) factors block column b+1: U1(b-1) (the last update of panel b-1 that touches it) and U2(b-2) must be done
      if (b >= 1 && have_u1[(b - 1) & 1]) VGG_CUDA_CHECK(cudaStreamWaitEvent(st, cs->ev_upd[(b - 1) & 1], 0));
      if (b >= 2 && have_u2[(b - 2) % 3]) VGG_CUDA_CHECK(cudaStreamWaitEvent(st, cs->ev_bulk[(b - 2) % 3], 0));
      if ((rc = panel(b + 1))) return rc;
    }
    // join whatever the last two panels left on the side streams (capture needs every forked stream back)
    for (int i = 0; i < 2; ++i)
      if (have_u1[i]) VGG_CUDA_CHECK(cudaStreamWaitEvent(st, cs->ev_upd[i], 0));
    for (int i = 0; i < 3; ++i)
      if (have_u2[i]) VGG_CUDA_CHECK(cudaStreamWaitEvent(st, cs->ev_bulk[i], 0));
    return VGG_OK;
  }
  for (int b = 0; b + 1 < nblk; ++b) {
    const int k0 = b * CB, t0 = k0 + CB;
    const int T = (n - t0 + CT - 1) / CT;
    chol_update_kernel<<<T * (T + 1) / 2, C_THREADS, smem_u, st>>>(n, lda, k0, t0, 0, A, n, n, 0);
    VGG_LAUNCH_CHECK();
    if ((rc = panel(b + 1))) return rc;
  }
  return VGG_OK;
}

}  // namespace

// In-place Cholesky of the row-major lower triangle of A[n x n] (lda even, A 16-byte aligned): on return the lower
// triangle holds L and the strict upper triangle L^T.  info (device int): 0 or the 1-based index of the first
// non-positive pivot.
int chol_lower_inplace(int n, int lda, double* A, double* Ldiag, int* info, cudaStream_t st) {
  VGG_REQUIRE((lda % 2) == 0, "lda must be even");
  int rc;
  if ((rc = chol_set_attrs())) return rc;
  VGG_CUDA_CHECK(cudaMemsetAsync(info, 0, sizeof(int), st));
  const int nblk0 = (n + CB - 1) / CB;
  int* flags = reinterpret_cast<int*>(Ldiag + (size_t)nblk0 * CB * CB);
  VGG_CUDA_CHECK(cudaMemsetAsync(flags, 0, sizeof(int) * (size_t)nblk0, st));
  const int nblk = (n + CB - 1) / CB;
  CholStreams* cs = nullptr;
  if ((rc = chol_streams(&cs))) return rc;
  if (nblk < 3) return chol_enqueue(n, lda, A, Ldiag, info, flags, st, cs);
  // one captured graph per (matrix, order): ~60 launches + events become a single cudaGraphLaunch
  typedef std::tuple<double*, int, int, int*, double*, unsigned long long> Key;
  static thread_local std::map<Key, cudaGraphExec_t> cache;
  unsigned long long band_hash = (unsigned long long)g_chol_arrow_blk;
  for (int v : g_chol_band_end) band_hash = band_hash * 1000003ull + (unsigned long long)(v + 1);
  const Key key(A, n, lda, info, Ldiag, band_hash);
  auto it = cache.find(key);
  if (it == cache.end()) {
    const long long launches_before = g_launch_count;
    cudaGraph_t graph = nullptr;
    VGG_CUDA_CHECK(cudaStreamBeginCapture(cs->cap, cudaStreamCaptureModeThreadLocal));
    rc = chol_enqueue(n, lda, A, Ldiag, info, flags, cs->cap, cs);
    const cudaError_t ce = cudaStreamEndCapture(cs->cap, &graph);
    g_launch_count = launches_before;
    if (rc) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    VGG_CUDA_CHECK(ce);
    cudaGraphExec_t exec = nullptr;
    VGG_CUDA_CHECK(cudaGraphInstantiate(&exec, graph, 0));
    cudaGraphDestroy(graph);
    if (cache.size() > 8) {
      for (auto& kv : cache) cudaGraphExecDestroy(kv.second);
      cache.clear();
    }
    it = cache.emplace(key, exec).first;
  }
  VGG_CUDA_CHECK(cudaGraphLaunch(it->second, st));
  g_launch_count += 1 + 3 * (nblk - 1);          // kernels inside the graph (upper bound: the last panels have no bulk update)
  return VGG_OK;
}

}  // namespace vgg

// tools/microbench.py chol128: one CTA, POTRF128 of A (host, row-major SPD 128 x 128), cycles per phase
extern "C" int vgg_dev_chol128_probe(int reps, const double* A_host, double* L_host, long long* prof13_host) {
  using namespace vgg;
  VGG_REQUIRE(A_host && L_host && prof13_host && reps > 0, "chol128 probe: bad arguments");
  double *dA = nullptr, *dL = nullptr;
  long long* dP = nullptr;
  VGG_CUDA_CHECK(cudaMalloc(&dA, sizeof(double) * CB * CB));
  VGG_CUDA_CHECK(cudaMalloc(&dL, sizeof(double) * CB * CB));
  VGG_CUDA_CHECK(cudaMalloc(&dP, sizeof(long long) * 13));
  VGG_CUDA_CHECK(cudaMemcpy(dA, A_host, sizeof(double) * CB * CB, cudaMemcpyHostToDevice));
  VGG_CUDA_CHECK(cudaMemset(dP, 0, sizeof(long long) * 13));
  const int smem = (int)(sizeof(double) * (CB + C_RPC) * CLD);
  VGG_CUDA_CHECK(cudaFuncSetAttribute(chol128_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  chol128_probe_kernel<<<1, C_THREADS, smem>>>(dA, dL, dP, reps, C_RPC);
  VGG_LAUNCH_CHECK();
  VGG_CUDA_CHECK(cudaDeviceSynchronize());
  VGG_CUDA_CHECK(cudaMemcpy(L_host, dL, sizeof(double) * CB * CB, cudaMemcpyDeviceToHost));
  VGG_CUDA_CHECK(cudaMemcpy(prof13_host, dP, sizeof(long long) * 13, cudaMemcpyDeviceToHost));
  cudaFree(dA);
  cudaFree(dL);
  cudaFree(dP);
  return VGG_OK;
}

// tests: install / clear (count = 0) the block structure the next factorisations assume (csrc/ba_solve.cu sets the same
// globals from the visibility mask for the duration of a solve)
extern "C" int vgg_dev_set_chol_band(const int* end_blk_host, int count, int arrow_blk) {
  using namespace vgg;
  g_chol_band_end.assign(end_blk_host, end_blk_host + (count > 0 ? count : 0));
  g_chol_arrow_blk = count > 0 ? arrow_blk : 0;
  return VGG_OK;
}

