// Fused reprojection residual + analytic Jacobian + normal-equation block kernel.
//
// Replaces, per LM iteration, what Ceres does on the CPU for the reference: evaluate COLMAP's
// ReprojErrorCostFunction<SimplePinhole|SimpleRadial> for every observation with autodiff Jets and
// hand the 2x(dc+3) Jacobians to the Schur eliminator (reached from
// vggsfm/utils/triangulation.py:213,1050,1142 through pycolmap.bundle_adjustment).
//
// Mapping (round-1 profile: the first version -- one thread per track, camera blocks reduced across the
// warp every frame -- spent 543 of 870 warp instructions per observation row on shuffles/selects, not on
// FP64 math).  Now one LANE owns one FRAME and a warp marches over tracks:
//   * the per-camera blocks (g_c, H_cc upper-packed, H_cs: 27..44 doubles) accumulate in the lane's
//     REGISTERS over the warp's whole track range and are flushed once with f64 REDs -- no per-observation
//     cross-lane traffic for them at all;
//   * the per-point blocks (g_p, H_pp, shared-intrinsics coupling: 9..15 doubles) go through a small per-warp
//     shared-memory scratch (one column per lane): 9..15 lanes each sum one row of 32 and commit it with one
//     RED instruction -- this keeps them out of the register file, which the camera accumulators fill;
//   * the coupling block W = J_c^T J_p lives in a TRACK-MAJOR layout W[n][row][3] (row = s*dc+i), so the 32
//     lanes' blocks of one track are 32*dc*24 B CONTIGUOUS bytes: each warp stages them in shared memory
//     (16-byte stores) and ships them with ONE TMA bulk store per track (cp.async.bulk.global.shared::cta ->
//     UBLKCP), double buffered against the next track's math.  W is 94 % of the kernel's HBM traffic.  The
//     track-major layout also makes the Schur operand build and the back-substitution transpose-free
//     (ba_schur.cu).
//   * observations (uv 8 B + mask 1 B) are read with 32-byte vector loads, 4 tracks per lane at a time,
//     prefetched one batch ahead; poses/intrinsics sit transposed in shared memory (one frame per lane).
// Algorithmic HBM bytes per observation: 9 + 24*dc (+ amortised per-frame/per-point terms), see DESIGN.md.
#include <utility>
#include "common.cuh"
#include "dev_probes.h"

namespace vgg {

// kernel-only timing for bench.py's roofline (csrc/dev_probes.h): an event pair on the launching stream, directly
// around the ba_blocks_kernel launch (the accumulator memsets stay outside)
extern BandDev g_band_dev;         // csrc/ba_schur.cu
static bool g_blocks_timing = false;
static cudaEvent_t g_blocks_ev[2] = {nullptr, nullptr};

constexpr int BW = 4;            // warps per CTA
constexpr int BT = BW * 32;      // threads per CTA
constexpr int TB = 4;            // tracks per prefetch batch (32 B of uv per lane)
constexpr int XT = 32;           // tracks per shared-memory point tile (one per lane)
constexpr int PVS = 33;          // row stride of the per-point scratch (odd: conflict-free column sums)

template <int MODEL, int MODE>
struct BlkCfg {
  static constexpr int NI = (MODEL == VGG_SIMPLE_PINHOLE) ? 1 : 2;
  static constexpr int DC = (MODE == VGG_INTR_PER_FRAME) ? 6 + NI : 6;
  static constexpr int NS = (MODE == VGG_INTR_SHARED) ? NI : 0;
  static constexpr int NPACK = DC * (DC + 1) / 2;
  static constexpr int KR = DC + NPACK + 6 * NS;   // per-frame camera record length
  static constexpr int NP = 9 + 3 * NS;            // per-point reduced values: g_p 3, H_pp 6, W_s 3*NS
};

// ---- compile-time layout of the per-frame camera record: g_c[DC] | H_cc upper-packed | H_cs[6][NS] ----
__host__ __device__ constexpr int pack_row(int dc, int p) {
  int i = 0;
  while (p >= dc - i) { p -= dc - i; ++i; }
  return i;
}
__host__ __device__ constexpr int pack_col(int dc, int p) {
  int i = 0;
  while (p >= dc - i) { p -= dc - i; ++i; }
  return i + p;
}

template <int DC, int NS, int K, int KR>
__device__ __forceinline__ void cam_accumulate_one(double (&acc)[KR], const double* jc0, const double* jc1, double rx,
                                                   double ry) {
  constexpr int NPACK = DC * (DC + 1) / 2;
  if constexpr (K < DC) {
    acc[K] = fma(jc0[K], rx, fma(jc1[K], ry, acc[K]));
  } else if constexpr (K < DC + NPACK) {
    constexpr int i = pack_row(DC, K - DC), j = pack_col(DC, K - DC);
    acc[K] = fma(jc0[i], jc0[j], fma(jc1[i], jc1[j], acc[K]));
  } else {
    constexpr int q = K - DC - NPACK;
    constexpr int i = q / (NS > 0 ? NS : 1), j = q % (NS > 0 ? NS : 1);
    acc[K] = fma(jc0[i], jc0[6 + j], fma(jc1[i], jc1[6 + j], acc[K]));
  }
}
template <int DC, int NS, int KR, int... K>
__device__ __forceinline__ void cam_accumulate(double (&acc)[KR], const double* jc0, const double* jc1, double rx,
                                               double ry, std::integer_sequence<int, K...>) {
  (cam_accumulate_one<DC, NS, K, KR>(acc, jc0, jc1, rx, ry), ...);
}

// One observation, branch-free: residual and Jacobian columns, all scaled by the validity mask (an invalid
// observation computes on a safe depth and contributes exact zeros).  jc: delta(3), t(3), f, k; jx: point(3).
template <int MODEL>
__device__ __forceinline__ void obs_math(const double* pw, int lane, const double* xt, float ox, float oy, bool valid,
                                         double* jc0, double* jc1, double* jx0, double* jx1, double& rx, double& ry) {
  const double2 xa = *reinterpret_cast<const double2*>(xt);
  const double2 xb = *reinterpret_cast<const double2*>(xt + 2);
  const double X0 = xa.x, X1 = xa.y, X2 = xb.x;
  const double m = valid ? 1.0 : 0.0;
  const double mp = (xb.y != 0.0) ? 0.0 : m;                    // constant point: no point columns
  const double R00 = pw[0 * 32 + lane], R01 = pw[1 * 32 + lane], R02 = pw[2 * 32 + lane], t0_ = pw[3 * 32 + lane];
  const double R10 = pw[4 * 32 + lane], R11 = pw[5 * 32 + lane], R12 = pw[6 * 32 + lane], t1_ = pw[7 * 32 + lane];
  const double R20 = pw[8 * 32 + lane], R21 = pw[9 * 32 + lane], R22 = pw[10 * 32 + lane], t2_ = pw[11 * 32 + lane];
  const double fo = pw[12 * 32 + lane], cx = pw[13 * 32 + lane], cy = pw[14 * 32 + lane];
  const double kk = (MODEL == VGG_SIMPLE_RADIAL) ? pw[15 * 32 + lane] : 0.0;
  const double a1 = R00 * X0 + R01 * X1 + R02 * X2;
  const double a2 = R10 * X0 + R11 * X1 + R12 * X2;
  const double a3 = R20 * X0 + R21 * X1 + R22 * X2;
  const double px = a1 + t0_, py = a2 + t1_;
  const double pz = valid ? (a3 + t2_) : 1.0;
  const double iz = 1.0 / pz;
  const double u = px * iz, w_ = py * iz;
  const double r2 = u * u + w_ * w_;
  const double d = 1.0 + kk * r2;
  rx = valid ? (fo * d * u + cx - (double)ox) : 0.0;            // select, not multiply: ox/oy of a masked slot may be anything
  ry = valid ? (fo * d * w_ + cy - (double)oy) : 0.0;
  double a00, a01, a11;
  if (MODEL == VGG_SIMPLE_RADIAL) {
    a00 = fo * (d + 2.0 * kk * u * u);
    a01 = fo * (2.0 * kk * u * w_);
    a11 = fo * (d + 2.0 * kk * w_ * w_);
  } else {
    a00 = fo; a01 = 0.0; a11 = fo;
  }
  // Jproj (2x3) = f*A * iz*[[1,0,-u],[0,1,-v]], masked
  const double izm = iz * m;
  const double j00 = a00 * izm, j01 = a01 * izm, j02 = -(a00 * u + a01 * w_) * izm;
  const double j10 = a01 * izm, j11 = a11 * izm, j12 = -(a01 * u + a11 * w_) * izm;
  const double b1 = 2.0 * a1, b2 = 2.0 * a2, b3 = 2.0 * a3;
  jc0[0] = b2 * j02 - b3 * j01;  jc1[0] = b2 * j12 - b3 * j11;
  jc0[1] = b3 * j00 - b1 * j02;  jc1[1] = b3 * j10 - b1 * j12;
  jc0[2] = b1 * j01 - b2 * j00;  jc1[2] = b1 * j11 - b2 * j10;
  jc0[3] = j00; jc0[4] = j01; jc0[5] = j02;
  jc1[3] = j10; jc1[4] = j11; jc1[5] = j12;
  jc0[6] = m * d * u;            jc1[6] = m * d * w_;
  jc0[7] = m * fo * u * r2;      jc1[7] = m * fo * w_ * r2;
  const double mq = (xb.y != 0.0) ? 0.0 : 1.0;
  jx0[0] = mq * (j00 * R00 + j01 * R10 + j02 * R20);
  jx0[1] = mq * (j00 * R01 + j01 * R11 + j02 * R21);
  jx0[2] = mq * (j00 * R02 + j01 * R12 + j02 * R22);
  jx1[0] = mq * (j10 * R00 + j11 * R10 + j12 * R20);
  jx1[1] = mq * (j10 * R01 + j11 * R11 + j12 * R21);
  jx1[2] = mq * (j10 * R02 + j11 * R12 + j12 * R22);
  (void)mp;
}

// coupling block (DC rows x 3, 16-byte stores into the staging buffer) and per-point values (scratch column)
template <int DC, int NS, int WB>
__device__ __forceinline__ void emit_blocks(double* wt, double* pvw, int lane, const double* jc0, const double* jc1,
                                            const double* jx0, const double* jx1, double rx, double ry) {
  double wb[WB];
#pragma unroll
  for (int i = 0; i < DC; ++i)
#pragma unroll
    for (int c = 0; c < 3; ++c) wb[i * 3 + c] = jc0[i] * jx0[c] + jc1[i] * jx1[c];
  if ((WB & 1) == 0) {
#pragma unroll
    for (int e = 0; e < WB; e += 2) *reinterpret_cast<double2*>(wt + e) = make_double2(wb[e], wb[e + 1]);
  } else {
#pragma unroll
    for (int e = 0; e < WB; ++e) wt[e] = wb[e];
  }
  pvw[0 * PVS + lane] = jx0[0] * rx + jx1[0] * ry;
  pvw[1 * PVS + lane] = jx0[1] * rx + jx1[1] * ry;
  pvw[2 * PVS + lane] = jx0[2] * rx + jx1[2] * ry;
  pvw[3 * PVS + lane] = jx0[0] * jx0[0] + jx1[0] * jx1[0];
  pvw[4 * PVS + lane] = jx0[0] * jx0[1] + jx1[0] * jx1[1];
  pvw[5 * PVS + lane] = jx0[0] * jx0[2] + jx1[0] * jx1[2];
  pvw[6 * PVS + lane] = jx0[1] * jx0[1] + jx1[1] * jx1[1];
  pvw[7 * PVS + lane] = jx0[1] * jx0[2] + jx1[1] * jx1[2];
  pvw[8 * PVS + lane] = jx0[2] * jx0[2] + jx1[2] * jx1[2];
#pragma unroll
  for (int j = 0; j < NS; ++j)
#pragma unroll
    for (int c = 0; c < 3; ++c) pvw[(9 + j * 3 + c) * PVS + lane] = jc0[6 + j] * jx0[c] + jc1[6 + j] * jx1[c];
}

// W row pitch (rows of 3 doubles) of one track: D rounded up to even so every track starts 16-B aligned
__host__ __device__ inline size_t w_pitch(int D) { return (size_t)(D + (D & 1)); }

template <int MODEL, int MODE, bool USE_TMA, int MINB>
__global__ void __launch_bounds__(BT, MINB) ba_blocks_kernel(
    int S, int N, int tracks_per_warp, const float* __restrict__ uv, const uint8_t* __restrict__ mask,
    const double* __restrict__ poses, const double* __restrict__ intr, const double* __restrict__ points,
    const uint8_t* __restrict__ point_const, double* __restrict__ cost, double* __restrict__ camrec,
    double* __restrict__ g_p, double* __restrict__ H_pp, double* __restrict__ W, double* __restrict__ shared_out,
    const int* __restrict__ fg_tracks) {
  using C = BlkCfg<MODEL, MODE>;
  constexpr int DC = C::DC, NS = C::NS, KR = C::KR, NP = C::NP;
  constexpr int WB = DC * 3;                       // doubles per observation block
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // per warp: pose/intrinsics transposed [16][32], two W staging buffers [32][WB]
  double* sm_pose = reinterpret_cast<double*>(smem_raw);                // [BW][16][32]
  double* sm_x = sm_pose + BW * 16 * 32;                                 // [BW][XT][4]: X,Y,Z,const flag per track
  double* sm_pv = sm_x + BW * XT * 4;                                    // [BW][2 tracks x 16][PVS]: per-point values, one column per lane
  double* sm_w = sm_pv + BW * 32 * PVS;                                  // [BW][2][32*WB]
  float* sm_obs = reinterpret_cast<float*>(sm_w + (size_t)BW * 2 * 32 * WB);   // [BW][2 stages][32 lanes][12]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = S * DC + NS;
  const size_t pitch = w_pitch(D);
  // work item of this warp: frame group g (32 frames), track range [t_begin, t_end)
  // Consecutive warps take consecutive FRAME GROUPS of the same track chunk: the 13 groups of a chunk then write the 13
  // adjacent segments of the same tracks' W rows (57 KB contiguous per track) at about the same time, which keeps the
  // DRAM pages open.  (r02 A/B: giving a CTA's warps one frame group and four chunks instead -- to merge their camera
  // flushes -- cost 19 % at 400 x 131072: 4380 -> 3554 GB/s.)
  const int ngroups = (S + 31) / 32;
  const int wid = blockIdx.x * BW + warp;
  const int g = wid % ngroups;
  const int chunk = wid / ngroups;
  const int t_begin = (int)min((long long)N, (long long)chunk * tracks_per_warp);
  const int t_end = min(N, t_begin + tracks_per_warp);
  // banded (sequential) problems: none of this warp's tracks is visible in its 32 frames.  Their W blocks stay at the zero
  // the solver wrote once per solve, and z_build / backsub skip the same region (csrc/ba_solve.cu, compute_band_hint).
  if (fg_tracks && (t_end <= fg_tracks[2 * g] || t_begin >= fg_tracks[2 * g + 1])) return;
  const int s = g * 32 + lane;
  const bool frame_ok = s < S;
  const int nf = min(32, S - g * 32);              // frames of this group that exist
  double* pw = sm_pose + warp * 16 * 32;
  double* xw = sm_x + warp * XT * 4;
  double* pvw = sm_pv + warp * 32 * PVS;
  float* ow = sm_obs + (size_t)warp * 2 * 32 * 12 + lane * 12;           // this lane's slot, stage stride 32*12
  double* wbuf = sm_w + (size_t)warp * 2 * 32 * WB;

  // camera of this lane -> shared, transposed (conflict-free one-frame-per-lane reads)
#pragma unroll
  for (int i = 0; i < 12; ++i) pw[i * 32 + lane] = frame_ok ? poses[(size_t)s * 12 + i] : 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) pw[(12 + i) * 32 + lane] = frame_ok ? intr[(size_t)s * 4 + i] : 0.0;
  __syncwarp();

  double acc[KR];
#pragma unroll
  for (int i = 0; i < KR; ++i) acc[i] = 0.0;
  double cost_acc = 0.0, gs0 = 0.0, gs1 = 0.0, hss0 = 0.0, hss1 = 0.0, hss2 = 0.0;

  // observation prefetch: TB tracks (32 B of uv, 4 mask bytes) per lane per batch, one batch ahead, staged with
  // cp.async (LDGSTS) into the lane's private shared-memory slot so the loads cannot be sunk next to their use
  // by the register allocator (r01 profile: 22 % of all stall samples sat on the first use of a register prefetch)
  const bool vec_ok = (N & 3) == 0;
  auto fetch = [&](int t0, int stage) {
    float* slot = ow + stage * 32 * 12;
    if (frame_ok && t0 < t_end) {
      const size_t o = (size_t)s * N + t0;
      if (vec_ok && t0 + TB <= t_end) {
        cp_async16(slot, uv + o * 2);
        cp_async16(slot + 4, uv + o * 2 + 4);
        cp_async4(slot + 8, mask + o);
      } else {
        uint32_t m = 0;
        for (int k = 0; k < TB; ++k) {
          const bool in = t0 + k < t_end;
          slot[2 * k] = in ? uv[(o + k) * 2] : 0.f;
          slot[2 * k + 1] = in ? uv[(o + k) * 2 + 1] : 0.f;
          if (in) m |= (uint32_t)(mask[o + k] != 0) << (8 * k);
        }
        reinterpret_cast<uint32_t*>(slot)[8] = m;
      }
    } else {
      *reinterpret_cast<float4*>(slot) = make_float4(0.f, 0.f, 0.f, 0.f);
      *reinterpret_cast<float4*>(slot + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      reinterpret_cast<uint32_t*>(slot)[8] = 0u;
    }
    cp_async_commit();
  };
  fetch(t_begin, 0);
  int batch = 0;
  for (int t0 = t_begin; t0 < t_end; t0 += TB) {
    if (((t0 - t_begin) & (XT - 1)) == 0) {
      // next 32 tracks' points -> shared (one track per lane, coalesced), read back as broadcasts
      __syncwarp();
      const int nn = t0 + lane;
      double x0 = 0.0, x1 = 0.0, x2 = 1.0, cf = 1.0;
      if (nn < t_end) {
        x0 = points[(size_t)nn * 3]; x1 = points[(size_t)nn * 3 + 1]; x2 = points[(size_t)nn * 3 + 2];
        cf = (point_const && point_const[nn] != 0) ? 1.0 : 0.0;
      }
      *reinterpret_cast<double2*>(xw + lane * 4) = make_double2(x0, x1);
      *reinterpret_cast<double2*>(xw + lane * 4 + 2) = make_double2(x2, cf);
      __syncwarp();
    }
    fetch(t0 + TB, (batch + 1) & 1);                              // next batch in flight during this one
    cp_async_wait<1>();                                           // ... and the current one has landed
    const float* cur = ow + (batch & 1) * 32 * 12;
    const float4 ca = *reinterpret_cast<const float4*>(cur);
    const float4 cb = *reinterpret_cast<const float4*>(cur + 4);
    const uint32_t cm = reinterpret_cast<const uint32_t*>(cur)[8];
    ++batch;
#pragma unroll 1
    for (int k = 0; k < TB; k += 2) {                            // two tracks per step: one branch-free block
      const int nA = t0 + k;
      if (nA >= t_end) break;                                    // warp-uniform
      const bool hasB = nA + 1 < t_end;
      // ---- math for both tracks, registers only (overlaps the previous step's TMA read-out)
      double jcA0[8], jcA1[8], jxA0[3], jxA1[3], rxA, ryA;
      double jcB0[8], jcB1[8], jxB0[3], jxB1[3], rxB, ryB;
      {
        const float ox = k == 0 ? ca.x : cb.x, oy = k == 0 ? ca.y : cb.y;
        const bool valid = frame_ok && ((cm >> (8 * k)) & 0xffu) != 0;
        obs_math<MODEL>(pw, lane, xw + ((nA - t_begin) & (XT - 1)) * 4, ox, oy, valid, jcA0, jcA1, jxA0, jxA1, rxA, ryA);
      }
      {
        const float ox = k == 0 ? ca.z : cb.z, oy = k == 0 ? ca.w : cb.w;
        const bool valid = hasB && frame_ok && ((cm >> (8 * (k + 1))) & 0xffu) != 0;
        obs_math<MODEL>(pw, lane, xw + ((nA + 1 - t_begin) & (XT - 1)) * 4, ox, oy, valid, jcB0, jcB1, jxB0, jxB1, rxB, ryB);
      }
      cost_acc += 0.5 * (rxA * rxA + ryA * ryA) + 0.5 * (rxB * rxB + ryB * ryB);
      // ---- both staging buffers must have been read out by the previous step's bulk stores
      if (USE_TMA) {
        if (lane == 0) tma_store_wait_read<0>();
        __syncwarp();
      }
      double* wA = wbuf + lane * WB;
      double* wB = wbuf + 32 * WB + lane * WB;
      emit_blocks<DC, NS, WB>(wA, pvw, lane, jcA0, jcA1, jxA0, jxA1, rxA, ryA);
      emit_blocks<DC, NS, WB>(wB, pvw + 16 * PVS, lane, jcB0, jcB1, jxB0, jxB1, rxB, ryB);
      // ---- ship the 32 frames' blocks of each track: contiguous runs W[n][g*32*DC .. +nf*DC][3]
      double* dstA = W + ((size_t)nA * pitch + (size_t)g * 32 * DC) * 3;
      double* dstB = dstA + pitch * 3;
      const uint32_t bytes = (uint32_t)nf * WB * 8u;
      if (USE_TMA && (bytes & 15u) == 0) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_1d(dstA, wbuf, bytes);
          if (hasB) tma_store_1d(dstB, wbuf + 32 * WB, bytes);
          tma_store_commit();
        }
      } else {
        __syncwarp();
        for (int e = lane; e < nf * WB; e += 32) dstA[e] = wbuf[e];
        if (hasB)
          for (int e = lane; e < nf * WB; e += 32) dstB[e] = wbuf[32 * WB + e];
        __syncwarp();
      }
      // ---- camera records straight into registers
      cam_accumulate<DC, NS, KR>(acc, jcA0, jcA1, rxA, ryA, std::make_integer_sequence<int, KR>{});
      cam_accumulate<DC, NS, KR>(acc, jcB0, jcB1, rxB, ryB, std::make_integer_sequence<int, KR>{});
      if (NS > 0) {
        gs0 += jcA0[6] * rxA + jcA1[6] * ryA + jcB0[6] * rxB + jcB1[6] * ryB;
        hss0 += jcA0[6] * jcA0[6] + jcA1[6] * jcA1[6] + jcB0[6] * jcB0[6] + jcB1[6] * jcB1[6];
        if (NS > 1) {
          gs1 += jcA0[7] * rxA + jcA1[7] * ryA + jcB0[7] * rxB + jcB1[7] * ryB;
          hss1 += jcA0[6] * jcA0[7] + jcA1[6] * jcA1[7] + jcB0[6] * jcB0[7] + jcB1[6] * jcB1[7];
          hss2 += jcA0[7] * jcA0[7] + jcA1[7] * jcA1[7] + jcB0[7] * jcB0[7] + jcB1[7] * jcB1[7];
        }
      }
      // ---- per-point sums over the warp's frames: lanes 0..NP-1 take track A, lanes 16..16+NP-1 track B
      {
        const int v = lane & 15;
        const int nT = nA + (lane >> 4);
        double r = 0.0;
        if (v < NP) {
          const double* row = pvw + ((lane >> 4) * 16 + v) * PVS;
          double r0 = 0.0, r1 = 0.0, r2s = 0.0, r3 = 0.0;      // four independent chains, not one of 32
#pragma unroll
          for (int j = 0; j < 32; j += 4) { r0 += row[j]; r1 += row[j + 1]; r2s += row[j + 2]; r3 += row[j + 3]; }
          r = (r0 + r1) + (r2s + r3);
        }
        if (r != 0.0 && nT < t_end) {
          if (v < 3) atomicAdd(&g_p[(size_t)nT * 3 + v], r);
          else if (v < 9) atomicAdd(&H_pp[(size_t)nT * 6 + (v - 3)], r);
          else if (v < NP) atomicAdd(&W[((size_t)nT * pitch + (size_t)S * DC + (v - 9) / 3) * 3 + (v - 9) % 3], r);
        }
      }
      __syncwarp();        // the scratch and the staging buffers are rewritten next step
    }
  }
  if (USE_TMA && lane == 0) tma_store_wait_all<0>();

  // flush this lane's camera record
  if (frame_ok && t_begin < t_end) {
#pragma unroll
    for (int i = 0; i < KR; ++i)
      if (acc[i] != 0.0) atomicAdd(&camrec[(size_t)s * KR + i], acc[i]);
  }
  // scalars: cost, g_s, H_ss
  {
    double a[8] = {cost_acc, gs0, gs1, hss0, hss1, hss2, 0.0, 0.0};
    const double r = warp_reduce_scatter<8>(a, lane);
    if (lane == 0 && r != 0.0) atomicAdd(cost, r);
    else if (NS > 0 && lane >= 1 && lane < 6 && r != 0.0) atomicAdd(&shared_out[lane - 1], r);
  }
}

template <int MODEL, int MODE>
static int launch_blocks(const vgg_ba_problem* p, double* cost, double* camrec, double* g_p, double* H_pp,
                         double* W, double* shared_out, int tracks_per_warp, cudaStream_t stream, bool outputs_zeroed) {
  using C = BlkCfg<MODEL, MODE>;
  const int S = p->S, N = p->N;
  const int D = S * C::DC + C::NS;
  const size_t pitch = w_pitch(D);
  const size_t smem = sizeof(double) * (BW * 16 * 32 + BW * XT * 4 + BW * 32 * PVS + (size_t)BW * 2 * 32 * C::DC * 3) +
                      sizeof(float) * BW * 2 * 32 * 12;
  const bool tma_ok = ((reinterpret_cast<uintptr_t>(W) & 15) == 0);
  const int ngroups = (S + 31) / 32;
  if (tracks_per_warp <= 0 && g_band_dev.fg_tracks) {
    // banded (sequential) problems: most (frame group, track chunk) warps return at once, so the chunks must be small
    // enough for the few that do not to spread over the machine (r02 launch list at 1000 frames x 32 k points: with the
    // dense sizing ~220 warps of 500 tracks each did all the work, 0.43 ms; the visible part is 0.5 GB)
    tracks_per_warp = 64;
  }
  if (tracks_per_warp <= 0) {
    // Every warp does the same amount of work, so the grid must be a whole number of waves: resident warps =
    // SMs x CTAs/SM (occupancy query) x BW.  Pick the smallest wave count that keeps >= 32 tracks per warp
    // amortising the per-warp camera flush (32 x KR REDs), capped at 4 waves; tracks per warp multiple of TB.
    static int slots = 0;
    if (slots == 0) {
      int dev = 0, sms = 148, per_sm = 2;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
      // the occupancy query needs the opt-in shared-memory limit in place (r02: without it the query returned 0, the
      // grid was sized for ONE CTA per SM and the 400 x 4096 launch ran as a single wave of 147 CTAs, half the warps)
      cudaFuncSetAttribute(ba_blocks_kernel<MODEL, MODE, true, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ba_blocks_kernel<MODEL, MODE, true, 2>, BT, smem);
      if (per_sm < 1) per_sm = 1;
      slots = sms * per_sm;
    }
    const long wave_warps = (long)slots * BW;
    long best_tpw = N;
    for (int waves = 1; waves <= 4; ++waves) {
      long chunks = waves * wave_warps / ngroups;
      if (chunks < 1) chunks = 1;
      long tpw = (N + chunks - 1) / chunks;
      tpw = (tpw + TB - 1) / TB * TB;
      if (tpw < 32 && waves > 1) break;
      best_tpw = tpw;
      if (tpw <= 512) break;                    // enough parallel slack; more waves only add flush traffic
    }
    tracks_per_warp = (int)best_tpw;
  }
  const int chunks = (N + tracks_per_warp - 1) / tracks_per_warp;
  const long nwarps = (long)chunks * ngroups;
  const unsigned grid = (unsigned)((nwarps + BW - 1) / BW);
  if (!outputs_zeroed) {
    // the five accumulators: ONE memset when the caller carved them back to back in the order of csrc/ba_solve.cu's
    // workspace (cost | shared | camrec | g_p | H_pp, gaps < 256 B) -- vggsfm_b200.bundle_adjustment.build_blocks does
    const char* lo = reinterpret_cast<const char*>(cost);
    const char* hi = reinterpret_cast<const char*>(H_pp + (size_t)N * 6);
    const size_t payload = sizeof(double) * (1 + 8 + (size_t)S * C::KR + (size_t)N * 9);
    const bool packed = lo < reinterpret_cast<const char*>(shared_out) && shared_out < camrec && camrec < g_p && g_p < H_pp &&
                        hi > lo && (size_t)(hi - lo) <= payload + 5 * 256;
    if (packed) {
      VGG_CUDA_CHECK(cudaMemsetAsync(cost, 0, (size_t)(hi - lo), stream));
    } else {
      VGG_CUDA_CHECK(cudaMemsetAsync(cost, 0, sizeof(double), stream));
      VGG_CUDA_CHECK(cudaMemsetAsync(camrec, 0, sizeof(double) * (size_t)S * C::KR, stream));
      VGG_CUDA_CHECK(cudaMemsetAsync(g_p, 0, sizeof(double) * (size_t)N * 3, stream));
      VGG_CUDA_CHECK(cudaMemsetAsync(H_pp, 0, sizeof(double) * (size_t)N * 6, stream));
      VGG_CUDA_CHECK(cudaMemsetAsync(shared_out, 0, sizeof(double) * 8, stream));
    }
  }
  if (pitch > (size_t)S * C::DC) {
    // shared-intrinsics rows (accumulated with REDs) and the pitch padding row of every track
    const size_t tail = pitch - (size_t)S * C::DC;
    VGG_CUDA_CHECK(cudaMemset2DAsync(W + (size_t)S * C::DC * 3, pitch * 24, 0, tail * 24, (size_t)N, stream));
  }
  // Aligned W: MINB = 2 lets ptxas use ~250 registers (no spills, 8 warps/SM).  Unaligned W (no bulk copies) keeps the
  // MINB = 3 build (168 registers, 12 warps/SM, a few spills).
  if (g_blocks_timing) VGG_CUDA_CHECK(cudaEventRecord(g_blocks_ev[0], stream));
  if (tma_ok) {
    auto kern = ba_blocks_kernel<MODEL, MODE, true, 2>;
    VGG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, BT, smem, stream>>>(S, N, tracks_per_warp, p->uv, p->mask, p->poses, p->intr, p->points,
                                     p->point_const, cost, camrec, g_p, H_pp, W, shared_out, g_band_dev.fg_tracks);
  } else {
    auto kern = ba_blocks_kernel<MODEL, MODE, false, 3>;
    VGG_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, BT, smem, stream>>>(S, N, tracks_per_warp, p->uv, p->mask, p->poses, p->intr, p->points,
                                     p->point_const, cost, camrec, g_p, H_pp, W, shared_out, g_band_dev.fg_tracks);
  }
  VGG_LAUNCH_CHECK();
  if (g_blocks_timing) VGG_CUDA_CHECK(cudaEventRecord(g_blocks_ev[1], stream));
  return VGG_OK;
}

int ba_build_blocks(const vgg_ba_problem* p, double* cost, double* camrec, double* g_p, double* H_pp, double* W,
                    double* shared_out, int tracks_per_warp, cudaStream_t stream, bool outputs_zeroed) {
  const int key = p->camera_model * 3 + p->intr_mode;
  switch (key) {
    case 0: return launch_blocks<0, 0>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
    case 1: return launch_blocks<0, 1>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
    case 2: return launch_blocks<0, 2>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
    case 3: return launch_blocks<1, 0>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
    case 4: return launch_blocks<1, 1>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
    case 5: return launch_blocks<1, 2>(p, cost, camrec, g_p, H_pp, W, shared_out, tracks_per_warp, stream, outputs_zeroed);
  }
  set_error("bad camera_model/intr_mode %d/%d", p->camera_model, p->intr_mode);
  return VGG_EINVAL;
}

}  // namespace vgg

extern "C" int vgg_dev_blocks_timing(int enable) {
  using namespace vgg;
  if (enable && !g_blocks_ev[0]) {
    VGG_CUDA_CHECK(cudaEventCreate(&g_blocks_ev[0]));
    VGG_CUDA_CHECK(cudaEventCreate(&g_blocks_ev[1]));
  }
  g_blocks_timing = enable != 0;
  return VGG_OK;
}

extern "C" int vgg_dev_blocks_last_ms(double* ms) {
  using namespace vgg;
  VGG_REQUIRE(g_blocks_ev[0] && ms, "blocks timing was never enabled");
  VGG_CUDA_CHECK(cudaEventSynchronize(g_blocks_ev[1]));
  float f = 0.f;
  VGG_CUDA_CHECK(cudaEventElapsedTime(&f, g_blocks_ev[0], g_blocks_ev[1]));
  *ms = (double)f;
  return VGG_OK;
}
