// Schur SYRK on the 5th-generation tensor cores: Sraw -= Zt^T Zt in FP64-equivalent precision computed with
// INT8 tcgen05.mma (Ozaki splitting), the step SURVEY section 0.6 / DESIGN section 4.2 name as the dominant cost
// of a bundle-adjustment iteration (76.5 GFLOP at 400 x 4096; 2.46 ms on the FP64 pipe with DMMA).
//
// FP64 has no tcgen05 path on sm_100a, but INT8 does (kind::i8, 8192 MAC/clk/SM, exact int32 accumulation).
//   1. every column d of Z (a reduced camera parameter) gets a power-of-two scale 2^e_d >= max_k |Z[k][d]|;
//      x = Z 2^-e_d is rounded to B = 8s-2 fractional bits and written as s balanced base-256 digits
//      (int8 "slices", most significant first): x = 2^-B sum_p d_p 256^(s-p)          (oz_slice_kernel)
//   2. (Z^T Z)_ij = 2^(e_i+e_j-2B) sum_t 256^(2s-t) C_t,  C_t = sum_{p+q=t} sum_k d_p[k][i] d_q[k][j]:
//      every C_t is an exact int32 (|d| <= 128, at most 7 pairs and 16384 k per work item: |C_t| < 2^31); orders t > s+1 are below
//      the rounding of step 1 and are dropped, leaving s(s+1)/2 int8 GEMMs (28 for s = 7)  (oz_syrk_kernel)
//   3. the epilogue recombines the C_t of a tile in FP64 registers and adds -value into Sraw with f64 RED
//      (multimem.red or a remote RED in the multi-GPU modes).
//
// oz_syrk_kernel is a persistent, warp-specialised tcgen05 kernel (one CTA per SM):
//   warp 0   producer: the int8 slices are stored in HBM as 8 KB tile images that are already in the 64-byte
//            swizzled K-major shared-memory layout UMMA wants, so a tile is ONE 1-D bulk copy (cp.async.bulk ->
//            UBLKCP) completing on an mbarrier -- no tensor map, no driver API;
//   warp 1   MMA issuer: one thread issues tcgen05.mma.cta_group::1.kind::i8 (M=128, N=128, K=32) for every
//            (p,q) pair of the work item's order group into up to four 128-column TMEM accumulators (one per order
//            t), tcgen05.commit releases the smem stage / publishes the accumulators;
//   warps 2-9 epilogue: tcgen05.ld the accumulators, combine the orders in FP64 registers, release TMEM, then
//            scale by 2^(e_i+e_j) and RED into the lower triangle while the next item's MMAs already run.
// Work items (tile, order group, k range) are built on the host, longest first, and strided over the CTAs.
#include "common.cuh"
#include "dev_probes.h"

#include <algorithm>
#include <vector>

namespace vgg {

namespace {

constexpr int OZ_BM = 128;                       // tile rows (reduced camera parameters)
constexpr int OZ_BK = 64;                        // k bytes per block = one 64-byte swizzle atom
constexpr int OZ_TILE_BYTES = OZ_BM * OZ_BK;     // 8 KB
constexpr int OZ_STAGES = 2;
constexpr int OZ_STAGE_TILES = 14;
constexpr int OZ_STAGE_BYTES = OZ_STAGE_TILES * OZ_TILE_BYTES;   // 112 KB
constexpr int OZ_THREADS = 320;                  // producer warp, MMA warp, 8 epilogue warps
constexpr int OZ_MAX_PAIRS = 20;
constexpr int OZ_MAX_ITEM_KB = 256;               // k blocks per work item: 7 pairs x 128^2 x 256 x 64 < 2^31 (exact int32 accumulators)
constexpr int OZ_PREFETCH = 4;                   // k blocks of L2 prefetch distance ahead of the bulk copies
constexpr int OZ_MAX_GROUPS = 3;
constexpr int OZ_MAX_ACC = 4;                    // 128-column TMEM accumulators (orders) per group
constexpr int OZ_EXPO_BAD = INT32_MIN;           // column holds a non-finite value
constexpr size_t OZ_SMEM_BYTES = (size_t)OZ_STAGES * OZ_STAGE_BYTES + 1024 + 128;

struct OzGroup {
  int n_a, n_b, n_pairs, n_acc;
  int exp_base;                                  // 8 (2s - tmax) - 2B
  uint8_t a_slice[8], b_slice[8];                // slice held by tile slot i / n_a + i
  uint8_t pair_a[OZ_MAX_PAIRS], pair_b[OZ_MAX_PAIRS], pair_acc[OZ_MAX_PAIRS];
  uint8_t pair_b_diag[OZ_MAX_PAIRS];             // on diagonal tiles B_q is the A slot that holds slice q
  uint8_t acc_shift[4];                          // 8 (tmax - t) of accumulator a
};
struct OzPlan {
  int slices, n_groups;
  OzGroup g[OZ_MAX_GROUPS];
};
struct OzWork {
  int bi, bj, group, kb0, kb1;
};

// ---------------------------------------------------------------------------------------------------------
// 1. column scales
__global__ void oz_rowmax_kernel(int Kpad, int Dpad, int k_per, const double* __restrict__ Zt,
                                 unsigned long long* __restrict__ amax) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= Dpad) return;
  const int k0 = blockIdx.y * k_per, k1 = min(Kpad, k0 + k_per);
  double m = 0.0;
  bool bad = false;
  for (int k = k0; k < k1; ++k) {
    const double a = fabs(Zt[(size_t)k * Dpad + d]);
    bad |= !(a <= 1.7976931348623157e308);
    m = fmax(m, a);
  }
  if (bad) m = __longlong_as_double(0x7ff0000000000000LL);
  if (m > 0.0) atomicMax(&amax[d], (unsigned long long)__double_as_longlong(m));
}

// 2. slices, written as pre-swizzled 8 KB tile images: tile (slice p, row block rb, k block kb) holds rows
//    d = rb*128 + r, bytes k = kb*64 + kk at offset r*64 + (((kk >> 4) ^ ((r >> 1) & 3)) << 4) + (kk & 15)
//    (the 64-byte swizzle, Swizzle<2,4,3>, of a K-major 128 x 64 B tile whose base is 1024-byte aligned).
//    Balanced base-256 digits come from ONE 64-bit add: with X = rint(x 2^B), |X| <= 2^B, the bytes of
//    X + 0x80..80 (s bytes of 0x80) are d_p + 128, so d_p = byte ^ 0x80.  A warp owns 8 rows x 4 chunks: its loads are
//    4 x 64-byte segments per k and its stores 512 contiguous bytes per slice.
__global__ void __launch_bounds__(512) oz_slice_kernel(int Kpad, int Dpad, int KB, int s,
                                                       const double* __restrict__ Zt,
                                                       const unsigned long long* __restrict__ amax,
                                                       int* __restrict__ expo, double* __restrict__ pow2,
                                                       int8_t* __restrict__ slices, size_t slice_stride,
                                                       const int* __restrict__ kb_range /* [nb][2] or null */) {
  const int rb = blockIdx.x, kb = blockIdx.y;
  // banded problems (csrc/ba_solve.cu computes the ranges from the visibility mask): outside [lo, hi) this row block of Z
  // is zero and no work item reads its tile images
  const bool skip = kb_range && (kb < kb_range[2 * rb] || kb >= kb_range[2 * rb + 1]);
  const int r = (threadIdx.x >> 5) * 8 + ((threadIdx.x & 31) >> 2), cphys = threadIdx.x & 3;
  const int c = cphys ^ ((r >> 1) & 3);
  const int d = rb * OZ_BM + r;
  const double m = __longlong_as_double((long long)amax[d]);
  int e = 0;
  bool bad = false, zero = true;
  if (m > 0.0) {
    if (m <= 1.7976931348623157e308) {
      e = ilogb(m) + 1;
      zero = e < -900;                 // columns below 2^-900 are treated as exact zeros (keeps 2^(B-e) finite)
      if (zero) e = 0;
    } else {
      bad = true;
    }
  }
  if (kb == 0 && cphys == 0) {
    expo[d] = bad ? OZ_EXPO_BAD : e;
    pow2[d] = bad ? 0.0 : ldexp(1.0, e);
  }
  if (skip) return;
  const int B = 8 * s - 2;
  const double scale = (bad || zero) ? 0.0 : __longlong_as_double((long long)(1023 + B - e) << 52);   // 2^(B-e), exact
  const unsigned long long bias = 0x0080808080808080ull >> (8 * (7 - s));
  uint32_t dig[7][4];
#pragma unroll
  for (int p = 0; p < 7; ++p) dig[p][0] = dig[p][1] = dig[p][2] = dig[p][3] = 0u;
  const int kbase = kb * OZ_BK + c * 16;
  double z[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) z[i] = (kbase + i < Kpad) ? Zt[(size_t)(kbase + i) * Dpad + d] : 0.0;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const unsigned long long Y = ((unsigned long long)__double2ll_rn(z[i] * scale) + bias) ^ bias;   // byte j = digit of 256^j
    const uint32_t lo = (uint32_t)Y, hi = (uint32_t)(Y >> 32);
#pragma unroll
    for (int p = 0; p < 7; ++p) {
      if (p < s) {
        const int j = s - 1 - p;                           // slice p (most significant first) is byte j
        const uint32_t byte = ((j < 4 ? lo >> (8 * j) : hi >> (8 * (j - 4))) & 255u);
        dig[p][i >> 2] |= byte << (8 * (i & 3));
      }
    }
  }
  const size_t off = ((size_t)rb * KB + kb) * OZ_TILE_BYTES + (size_t)r * OZ_BK + (size_t)(cphys << 4);
#pragma unroll
  for (int p = 0; p < 7; ++p)
    if (p < s) *reinterpret_cast<uint4*>(slices + (size_t)p * slice_stride + off) = make_uint4(dig[p][0], dig[p][1], dig[p][2], dig[p][3]);
}

// ---------------------------------------------------------------------------------------------------------
// tcgen05 / TMEM helpers (PTX ISA 8.6+, sm_100a)
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, int8 x int8 -> int32, M = 128, N = 128, K = 32
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand in tensor memory (128 lanes = rows, 8 32-bit columns = 32 int8 of K per row): the MMA then
// reads only B from shared memory (oz_mma_rate_kernel)
__device__ __forceinline__ void umma_i8_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// pull a global range into L2 ahead of the bulk copy that will read it (hides the HBM latency of first-touch tiles)
__device__ __forceinline__ void l2_prefetch(const void* gptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
// shared-memory matrix descriptor: K-major, 64-byte swizzle, 8-row atoms 512 B apart, sm_100 descriptor version
__device__ __forceinline__ uint64_t smem_desc_sw64(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(512 >> 4) << 32) | (1ull << 46) | (4ull << 61);
}
// instruction descriptor: D = s32, A = B = signed int8, both K-major, N = 128, M = 128
constexpr uint32_t OZ_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// ---------------------------------------------------------------------------------------------------------
// 3. persistent tcgen05 SYRK
// Two variants were measured slower on a B200 and removed (profiles/README.md): the A operand staged in tensor memory by
// four extra warps (exact, 1.86 ms per call against 1.07 ms at 400 x 4096: the staging round per K = 32 half outlasts the
// ~15 MMAs it feeds) and CTA pairs issuing cta_group::2 MMAs with M = 256 (exact, 1.21 ms against 1.07 ms).
__global__ void __maxnreg__(168)                 // 320 threads x 168 registers
    oz_syrk_kernel(const __grid_constant__ OzPlan plan, const OzWork* __restrict__ work, int nwork, int KB,
                   const int8_t* __restrict__ slices, size_t slice_stride, const int* __restrict__ expo,
                   const double* __restrict__ pow2, int Dpad, double* __restrict__ Cmat, ptrdiff_t mc_off,
                   const __grid_constant__ FabricDev fd) {
  extern __shared__ __align__(1024) uint8_t oz_smem[];
  uint8_t* tiles = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<size_t>(oz_smem), 1024));
  uint64_t* full = reinterpret_cast<uint64_t*>(tiles + (size_t)OZ_STAGES * OZ_STAGE_BYTES);
  uint64_t* empty = full + OZ_STAGES;
  uint64_t* tmem_full = empty + OZ_STAGES;
  uint64_t* tmem_empty = tmem_full + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < OZ_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tmem_full, 1);
    mbar_init(tmem_empty, 8);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===== producer =====
    if (lane == 0) {
      int stage = 0, phase = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x) {
        const OzWork wk = work[w];
        const OzGroup& g = plan.g[wk.group];
        const bool diag = wk.bi == wk.bj;
        for (int kb = wk.kb0; kb < wk.kb1; ++kb) {
          const int kpf = kb + OZ_PREFETCH;
          if (kpf < wk.kb1) {
            for (int i = 0; i < g.n_a; ++i)
              l2_prefetch(slices + (size_t)g.a_slice[i] * slice_stride + ((size_t)wk.bi * KB + kpf) * OZ_TILE_BYTES, OZ_TILE_BYTES);
            for (int i = 0; i < (diag ? 0 : g.n_b); ++i)
              l2_prefetch(slices + (size_t)g.b_slice[i] * slice_stride + ((size_t)wk.bj * KB + kpf) * OZ_TILE_BYTES, OZ_TILE_BYTES);
          }
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* dst = tiles + (size_t)stage * OZ_STAGE_BYTES;
          mbar_expect_tx(&full[stage], (uint32_t)(g.n_a + (diag ? 0 : g.n_b)) * OZ_TILE_BYTES);
          for (int i = 0; i < g.n_a; ++i)
            tma_load_1d(dst + (size_t)i * OZ_TILE_BYTES,
                        slices + (size_t)g.a_slice[i] * slice_stride + ((size_t)wk.bi * KB + kb) * OZ_TILE_BYTES,
                        OZ_TILE_BYTES, &full[stage]);
          for (int i = 0; i < (diag ? 0 : g.n_b); ++i)
            tma_load_1d(dst + (size_t)(g.n_a + i) * OZ_TILE_BYTES,
                        slices + (size_t)g.b_slice[i] * slice_stride + ((size_t)wk.bj * KB + kb) * OZ_TILE_BYTES,
                        OZ_TILE_BYTES, &full[stage]);
          if (++stage == OZ_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int stage = 0, phase = 0, it = 0;
      for (int w = blockIdx.x; w < nwork; w += gridDim.x, ++it) {
        const OzWork wk = work[w];
        const OzGroup& g = plan.g[wk.group];
        const bool diag = wk.bi == wk.bj;
        mbar_wait(tmem_empty, (uint32_t)((it & 1) ^ 1));
        tc_fence_after();
        uint32_t acc_used = 0;
        for (int kb = wk.kb0; kb < wk.kb1; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t base = smem_u32(tiles + (size_t)stage * OZ_STAGE_BYTES);
          for (int pr = 0; pr < g.n_pairs; ++pr) {
            const uint32_t a_addr = base + (uint32_t)g.pair_a[pr] * OZ_TILE_BYTES;
            const uint32_t b_addr = base + (uint32_t)(diag ? g.pair_b_diag[pr] : g.n_a + g.pair_b[pr]) * OZ_TILE_BYTES;
            const uint32_t acc = g.pair_acc[pr];
#pragma unroll
            for (int ks = 0; ks < OZ_BK / 32; ++ks) {
              umma_i8(tmem_base + acc * 128u, smem_desc_sw64(a_addr + ks * 32), smem_desc_sw64(b_addr + ks * 32),
                      OZ_IDESC, (acc_used >> acc) & 1u);
              acc_used |= 1u << acc;
            }
          }
          umma_commit(&empty[stage]);
          if (++stage == OZ_STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        umma_commit(tmem_full);
      }
    }
  } else {
    // ===== epilogue (8 warps: TMEM lane quarter = warp % 4, column half = (warp - 2) / 4) =====
    const int quarter = warp & 3, half = (warp - 2) >> 2;
    const int row_local = quarter * 32 + lane, col0 = half * 64;
    int it = 0;
    for (int w = blockIdx.x; w < nwork; w += gridDim.x, ++it) {
      const OzWork wk = work[w];
      const OzGroup& g = plan.g[wk.group];
      mbar_wait(tmem_full, (uint32_t)(it & 1));
      tc_fence_after();
      double acc[64];
#pragma unroll
      for (int j = 0; j < 64; ++j) acc[j] = 0.0;
      for (int a = 0; a < g.n_acc; ++a) {
        const double wgt = (double)(1ull << g.acc_shift[a]);
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) {
          uint32_t v[16];
          tmem_ld16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(a * 128 + col0 + c16 * 16), v);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[c16 * 16 + j] = fma((double)(int)v[j], wgt, acc[c16 * 16 + j]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tmem_empty);
      // scale and accumulate into Sraw
      const int r = wk.bi * OZ_BM + row_local;
      const int er = expo[r];
      const bool diag = wk.bi == wk.bj;
      // 2^(e_r + e_c + exp_base) as two exact multiplications while the exponents are tame, ldexp otherwise
      const bool tame = er != OZ_EXPO_BAD && er > -400 && er < 400;
      const double sr = tame ? __longlong_as_double((long long)(1023 + er + g.exp_base) << 52) : 0.0;
#pragma unroll
      for (int j = 0; j < 64; ++j) {
        const int col = wk.bj * OZ_BM + col0 + j;
        const int ec = expo[col];
        double v = acc[j];
        if (er == OZ_EXPO_BAD || ec == OZ_EXPO_BAD) v = __longlong_as_double(0x7ff8000000000000LL);
        else if (tame && ec > -400 && ec < 400) v = v * sr * pow2[col];
        else v = ldexp(v, er + ec + g.exp_base);
        if (v != 0.0) {
          // The work list holds UPPER tiles (bi <= bj): TMEM lane = r, so the 32 lanes of one RED instruction hit 32
          // consecutive addresses of row `col` -- the mirrored element (col, r) of the row-major LOWER triangle, which is
          // what csrc/chol.cu factors (fabric mode: one multimem op per element).
          if (!diag || col >= r) {
            const size_t off = (size_t)col * Dpad + r;
            if (fd.world > 1) {
              // reduce-scatter: row block wk.bj of the lower triangle lives on rank (wk.bj mod world) until the gather
              // (csrc/fabric.cu); one system-scope RED over NVLink per element, only into the owner's copy
              asm volatile("red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(fd.peer[wk.bj % fd.world] + off), "d"(-v) : "memory");
            } else if (mc_off) {
              asm volatile("multimem.red.relaxed.sys.global.add.f64 [%0], %1;" ::"l"(Cmat + off + mc_off), "d"(-v) : "memory");
            } else {
              atomicAdd(Cmat + off, -v);
            }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}


// ---------------------------------------------------------------------------------------------------------
// tensor-pipe rate probe (tools/syrk_i8_check.py rate): back-to-back kind::i8 MMAs on resident shared-memory tiles,
// cycles per MMA for the three shared-memory layouts / two N.  Data content is irrelevant.
__global__ void __launch_bounds__(128, 1) oz_mma_rate_kernel(int iters, int mode, long long* out) {
  extern __shared__ __align__(1024) uint8_t oz_smem[];
  uint8_t* tiles = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<size_t>(oz_smem), 1024));
  __shared__ uint64_t bar;
  __shared__ uint32_t tptr;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    mbar_fence_init();
  }
  for (int i = threadIdx.x; i < 65536 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(tiles)[i] = 0x01010101u;
  fence_proxy_async();
  if (threadIdx.x < 32) tmem_alloc(&tptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = tptr;
  if (threadIdx.x == 0) {
    const uint32_t base = smem_u32(tiles);
    const int n = (mode & 1) ? 256 : 128;
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
    const int layout = (mode >> 1) & 3;      // 0: SW64 (64 B rows), 1: SW128 (128 B rows), 2: no swizzle
    const bool a_tmem = (mode & 8) != 0;     // A operand from tensor memory (columns 384..), B from shared memory
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
      const uint32_t a = base + (uint32_t)(it & 1) * 32, b = base + 32768 + (uint32_t)(it & 1) * 32;
      uint64_t da, db;
      if (layout == 0) {
        da = smem_desc_sw64(a); db = smem_desc_sw64(b);
      } else if (layout == 1) {
        da = (uint64_t)((a >> 4) & 0x3FFF) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
        db = (uint64_t)((b >> 4) & 0x3FFF) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
      } else {
        da = (uint64_t)((a >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
        db = (uint64_t)((b >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
      }
      if (a_tmem) umma_i8_ts(tb, tb + 384u + (uint32_t)(it & 1) * 8u, db, idesc, 1u);
      else umma_i8(tb, da, db, idesc, 1u);
    }
    umma_commit(&bar);
    mbar_wait(&bar, 0);
    out[0] = clock64() - t0;
  }
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tb, 512);
}

// ---------------------------------------------------------------------------------------------------------
// host side: order groups and work list
bool build_plan(int s, OzPlan* plan) {
  if (s < 3 || s > 7) return false;
  plan->slices = s;
  const int B = 8 * s - 2;
  const int tlast = s + 1;                       // orders 2 .. s+1 are kept
  int ng = 0;
  for (int t0 = 2; t0 <= tlast; t0 += OZ_MAX_ACC) {
    if (ng >= OZ_MAX_GROUPS) return false;
    OzGroup& g = plan->g[ng++];
    const int t1 = std::min(t0 + OZ_MAX_ACC - 1, tlast);
    g.n_acc = t1 - t0 + 1;
    g.exp_base = 8 * (2 * s - t1) - 2 * B;
    int slot_a[8], slot_b[8];
    for (int i = 0; i < 8; ++i) slot_a[i] = slot_b[i] = -1;
    g.n_a = g.n_b = g.n_pairs = 0;
    for (int t = t0; t <= t1; ++t) {
      g.acc_shift[t - t0] = (uint8_t)(8 * (t1 - t));
      for (int p = 1; p <= s; ++p) {
        const int q = t - p;
        if (q < 1 || q > s) continue;
        if (slot_a[p] < 0) {
          slot_a[p] = g.n_a;
          g.a_slice[g.n_a++] = (uint8_t)(p - 1);
        }
        if (slot_b[q] < 0) {
          slot_b[q] = g.n_b;
          g.b_slice[g.n_b++] = (uint8_t)(q - 1);
        }
        if (g.n_pairs >= OZ_MAX_PAIRS) return false;
        g.pair_a[g.n_pairs] = (uint8_t)slot_a[p];
        g.pair_b[g.n_pairs] = (uint8_t)slot_b[q];
        g.pair_acc[g.n_pairs] = (uint8_t)(t - t0);
        ++g.n_pairs;
      }
    }
    for (int pr = 0; pr < g.n_pairs; ++pr) {              // the order groups are symmetric in (p, q): slice q has an A slot
      const int q = g.b_slice[g.pair_b[pr]] + 1;
      if (slot_a[q] < 0) return false;
      g.pair_b_diag[pr] = (uint8_t)slot_a[q];
    }
    if (g.n_a + g.n_b > OZ_STAGE_TILES) return false;
  }
  plan->n_groups = ng;
  return true;
}


// Work items are handed out statically (item w goes to CTA w mod n, longest first), so the finishing time is
// the heaviest residue class.  The k-split granularity is chosen by simulating that assignment for a few candidate
// targets and keeping the best makespan (+ a small charge per item for its epilogue).
struct OzTileJob {
  int bi, bj;
  int kb0 = 0, kb1 = -1;       // k-block range in which BOTH row blocks can be non-zero (kb1 < 0: all of K)
};
void build_work_list(const OzPlan& plan, const std::vector<OzTileJob>& jobs, int KB, int nworkers,
                     std::vector<OzWork>* out) {
  long long total = 0, pairs_all = 0;
  for (int g = 0; g < plan.n_groups; ++g) pairs_all += plan.g[g].n_pairs;
  for (const OzTileJob& jb : jobs) total += pairs_all * (long long)((jb.kb1 < 0 ? KB : jb.kb1) - jb.kb0);
  const long long epilogue_cost = 24;            // pair-kblock equivalents of one item's TMEM drain + REDs (not overlapped part)
  long long best = -1;
  for (int div = 2; div <= 10; ++div) {
    const long long target = std::max<long long>(1, total / ((long long)nworkers * div));
    std::vector<std::pair<long long, OzWork>> items;
    for (const OzTileJob& jb : jobs) {
      const int jk0 = jb.kb0, jk1 = jb.kb1 < 0 ? KB : jb.kb1, len = jk1 - jk0;
      if (len <= 0) continue;
      for (int g = 0; g < plan.n_groups; ++g) {
        const long long cost = (long long)plan.g[g].n_pairs * len;
        int parts = (int)std::min<long long>(16, std::max<long long>(1, (cost + target / 2) / target));
        parts = std::max(parts, (len + OZ_MAX_ITEM_KB - 1) / OZ_MAX_ITEM_KB);      // int32 accumulators stay exact
        parts = std::min(parts, len);
        for (int p = 0; p < parts; ++p) {
          const int k0 = jk0 + (int)((long long)len * p / parts), k1 = jk0 + (int)((long long)len * (p + 1) / parts);
          items.push_back({(long long)plan.g[g].n_pairs * (k1 - k0), OzWork{jb.bi, jb.bj, g, k0, k1}});
        }
      }
    }
    std::stable_sort(items.begin(), items.end(), [](const auto& a, const auto& b) { return a.first > b.first; });
    std::vector<long long> load(nworkers, 0);
    for (size_t i = 0; i < items.size(); ++i) load[i % nworkers] += items[i].first + epilogue_cost;
    const long long makespan = *std::max_element(load.begin(), load.end());
    if (best < 0 || makespan < best) {
      best = makespan;
      out->clear();
      for (auto& it : items) out->push_back(it.second);
    }
  }
}

struct OzHostState {
  int Kpad = -1, Dpad = -1, slices = -1, sms = 0;
  std::vector<int> ranges;        // k-block range per row block the cached work list was built for (empty: dense)
  int* ranges_dev = nullptr;      // device copy for the slicing kernel
  size_t ranges_cap = 0;
  OzPlan plan;
  std::vector<OzWork> work;
  OzWork* pinned = nullptr;       // page-locked copy of `work`, so the per-call upload is a true async copy
  size_t pinned_cap = 0;
};

thread_local OzHostState g_oz;

int oz_max_parts(int KB) { return std::max(16, (KB + OZ_MAX_ITEM_KB - 1) / OZ_MAX_ITEM_KB); }

size_t oz_workspace_bytes(int Kpad, int Dpad, int s) {
  const int KB = (Kpad + OZ_BK - 1) / OZ_BK;
  const int nb = Dpad / OZ_BM;
  size_t bytes = 0;
  bytes += align_up((size_t)Dpad * 8, 256);                                   // amax
  bytes += align_up((size_t)Dpad * 4, 256);                                   // expo
  bytes += align_up((size_t)Dpad * 8, 256);                                   // pow2
  bytes += align_up((size_t)nb * (nb + 1) / 2 * OZ_MAX_GROUPS * oz_max_parts(KB) * sizeof(OzWork), 256);    // work list (upper bound)
  bytes += align_up((size_t)s * nb * KB * OZ_TILE_BYTES, 1024) + 1024;        // slices
  return bytes;
}

}  // namespace

size_t syrk_i8_workspace_bytes(int Kpad, int Dpad, int slices) { return oz_workspace_bytes(Kpad, Dpad, slices); }

// The column maxima can be produced by whoever writes Zt (z_build_kernel does): zero them with syrk_i8_reset_amax,
// hand syrk_i8_amax(ws) to the producer, then call launch_syrk_i8 with amax_ready = true.
unsigned long long* syrk_i8_amax(void* ws) { return static_cast<unsigned long long*>(ws); }
int syrk_i8_reset_amax(void* ws, int Dpad, cudaStream_t st) {
  VGG_CUDA_CHECK(cudaMemsetAsync(ws, 0, sizeof(unsigned long long) * Dpad, st));
  return VGG_OK;
}

// Sraw -= Zt^T Zt with s int8 slices.  Zt [Kpad][Dpad] (Dpad % 128 == 0), Cmat [Dpad][Dpad] row-major, LOWER triangle
// written.
// Band hint of the current solve (csrc/ba_solve.cu): [lo, hi) k-block range per 128-column row block of Zt outside which
// the block is exactly zero; empty = dense.  Tiles whose two ranges do not intersect are skipped, the others shortened.
std::vector<int> g_syrk_kb_ranges;
extern FabricDev g_fabric_dev;  // csrc/ba_schur.cu: reduce-scatter destinations of the current multi-GPU solve (world <= 1: off)

int launch_syrk_i8(int Kpad, int Dpad, const double* Zt, double* Cmat, ptrdiff_t mc_off, int s, void* ws,
                   size_t ws_bytes, cudaStream_t st, bool amax_ready) {
  VGG_REQUIRE(Dpad % OZ_BM == 0, "syrk_i8: Dpad must be a multiple of 128");
  VGG_REQUIRE(ws_bytes >= oz_workspace_bytes(Kpad, Dpad, s), "syrk_i8: workspace too small");
  const int KB = (Kpad + OZ_BK - 1) / OZ_BK;
  const int nb = Dpad / OZ_BM;
  OzHostState& hs = g_oz;
  const bool banded = (int)g_syrk_kb_ranges.size() == 2 * nb;
  if (hs.Kpad != Kpad || hs.Dpad != Dpad || hs.slices != s || (banded ? hs.ranges != g_syrk_kb_ranges : !hs.ranges.empty())) {
    hs.ranges = banded ? g_syrk_kb_ranges : std::vector<int>();
    if (banded) {
      if (hs.ranges_cap < hs.ranges.size()) {
        if (hs.ranges_dev) cudaFree(hs.ranges_dev);
        hs.ranges_cap = hs.ranges.size();
        VGG_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&hs.ranges_dev), sizeof(int) * hs.ranges_cap));
      }
      VGG_CUDA_CHECK(cudaMemcpyAsync(hs.ranges_dev, hs.ranges.data(), sizeof(int) * hs.ranges.size(), cudaMemcpyHostToDevice, st));
      VGG_CUDA_CHECK(cudaStreamSynchronize(st));          // the source is pageable host memory; once per (re)plan
    }
    VGG_REQUIRE(build_plan(s, &hs.plan), "syrk_i8: slices must be in [3,7]");
    int dev = 0;
    VGG_CUDA_CHECK(cudaGetDevice(&dev));
    VGG_CUDA_CHECK(cudaDeviceGetAttribute(&hs.sms, cudaDevAttrMultiProcessorCount, dev));
    VGG_CUDA_CHECK(cudaFuncSetAttribute(oz_syrk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)OZ_SMEM_BYTES));
    // work items: (tile, group, k range), longest first (build_work_list picks the k-split granularity)
    {
      std::vector<OzTileJob> jobs;
      for (int bi = 0; bi < nb; ++bi)
        for (int bj = 0; bj <= bi; ++bj) {                                    // upper tile (row block bj <= column block bi)
          OzTileJob jb{bj, bi};
          if (banded) {
            jb.kb0 = std::max(hs.ranges[2 * bi], hs.ranges[2 * bj]);
            jb.kb1 = std::min(hs.ranges[2 * bi + 1], hs.ranges[2 * bj + 1]);
            if (jb.kb1 <= jb.kb0) continue;
          }
          jobs.push_back(jb);
        }
      build_work_list(hs.plan, jobs, KB, hs.sms, &hs.work);
    }
    if (hs.work.size() > hs.pinned_cap) {
      if (hs.pinned) cudaFreeHost(hs.pinned);
      hs.pinned_cap = hs.work.size();
      VGG_CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&hs.pinned), sizeof(OzWork) * hs.pinned_cap, cudaHostAllocDefault));
    }
    std::copy(hs.work.begin(), hs.work.end(), hs.pinned);
    hs.Kpad = Kpad;
    hs.Dpad = Dpad;
    hs.slices = s;
  }
  Carver c(ws, ws_bytes);
  unsigned long long* amax = c.take<unsigned long long>(Dpad);
  int* expo = c.take<int>(Dpad);
  double* pow2 = c.take<double>(Dpad);
  OzWork* work_d = c.take<OzWork>((size_t)nb * (nb + 1) / 2 * OZ_MAX_GROUPS * oz_max_parts(KB));
  c.off = align_up(c.off, 1024);
  int8_t* slices = reinterpret_cast<int8_t*>(c.base + c.off);
  const size_t slice_stride = (size_t)nb * KB * OZ_TILE_BYTES;
  const int nwork = (int)hs.work.size();
  VGG_CUDA_CHECK(cudaMemcpyAsync(work_d, hs.pinned, sizeof(OzWork) * nwork, cudaMemcpyHostToDevice, st));
  if (!amax_ready) {
    VGG_CUDA_CHECK(cudaMemsetAsync(amax, 0, sizeof(unsigned long long) * Dpad, st));
    const int ksplit = 64;
    const int k_per = (Kpad + ksplit - 1) / ksplit;
    oz_rowmax_kernel<<<dim3(Dpad / 128, ksplit), 128, 0, st>>>(Kpad, Dpad, k_per, Zt, amax);
    VGG_LAUNCH_CHECK();
  }
  oz_slice_kernel<<<dim3(nb, KB), 512, 0, st>>>(Kpad, Dpad, KB, s, Zt, amax, expo, pow2, slices, slice_stride,
                                                banded ? hs.ranges_dev : nullptr);
  VGG_LAUNCH_CHECK();
  const int grid = std::min(hs.sms, nwork);
  oz_syrk_kernel<<<grid, OZ_THREADS, OZ_SMEM_BYTES, st>>>(hs.plan, work_d, nwork, KB, slices, slice_stride, expo, pow2, Dpad,
                                                          Cmat, mc_off, g_fabric_dev);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}

}  // namespace vgg

extern "C" {

/* development probe (csrc/dev_probes.h): install / clear (count = 0) the band hint the next SYRK calls plan with */
int vgg_dev_set_syrk_ranges(const int* ranges_host, int count) {
  using namespace vgg;
  g_syrk_kb_ranges.assign(ranges_host, ranges_host + (count > 0 ? count : 0));
  return VGG_OK;
}

int vgg_syrk_ozaki_workspace_bytes(int Kpad, int Dpad, int slices, size_t* bytes) {
  using namespace vgg;
  VGG_REQUIRE(bytes && Kpad > 0 && Dpad > 0 && Dpad % 128 == 0 && slices >= 3 && slices <= 7, "bad argument");
  *bytes = syrk_i8_workspace_bytes(Kpad, Dpad, slices);
  return VGG_OK;
}

/* cycles per tcgen05.mma.kind::i8 (M=128, K=32) issued back to back; mode bit0: N=256 instead of 128, mode>>1: smem
 * layout 0 = 64-byte swizzle, 1 = 128-byte swizzle, 2 = none.  out_cycles is a HOST pointer. */
int vgg_syrk_ozaki_mma_rate(int iters, int mode, double* out_cycles, void* stream) {
  using namespace vgg;
  g_launch_count = 0;
  VGG_REQUIRE(iters > 0 && out_cycles, "bad argument");
  long long* d = nullptr;
  VGG_CUDA_CHECK(cudaMalloc(&d, sizeof(long long)));
  VGG_CUDA_CHECK(cudaFuncSetAttribute(oz_mma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 66 * 1024 + 1024));
  oz_mma_rate_kernel<<<1, 128, 66 * 1024 + 1024, static_cast<cudaStream_t>(stream)>>>(iters, mode, d);
  VGG_LAUNCH_CHECK();
  long long h = 0;
  VGG_CUDA_CHECK(cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(d);
  *out_cycles = (double)h / iters;
  return VGG_OK;
}

int vgg_syrk_ozaki(int Kpad, int Dpad, const double* Zt, double* Cmat, int slices, void* workspace, size_t ws_bytes,
                   void* stream) {
  using namespace vgg;
  g_launch_count = 0;
  VGG_REQUIRE(Zt && Cmat && workspace, "null pointer");
  return launch_syrk_i8(Kpad, Dpad, Zt, Cmat, 0, slices, workspace, ws_bytes, static_cast<cudaStream_t>(stream), false);
}

}  // extern "C"
