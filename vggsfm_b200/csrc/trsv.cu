// Backward substitution U x = y for the reduced camera system (n = 2402 at 400 frames), one launch.
//
// After the bordered factorisation (csrc/ba_solve.cu) the forward substitution is already done; what is left is
// x = L^-T y.  The library call for it (cublasDtrsv, 0.24 ms at n = 2402) is bound by its dependency chain, not by the
// 23 MB it reads.  Here block row b (64 rows) belongs to CTA b of one co-resident grid (38 CTAs):
//   * every CTA inverts its 64 x 64 diagonal block in shared memory while it would otherwise wait (independent of x);
//   * it then walks the block columns j = last .. b+1: poll x_j itself (the output buffer is pre-filled with a sentinel
//     NaN pattern, so the data is its own flag: no fence, no second round trip), acc -= U[b][j] x_j, with the next tile
//     already in registers (tiles do not depend on x, only x_j does);
//   * x_b = inv(U_bb) acc (four threads per row), stored element-wise with volatile 8-byte stores.
// Block rows are handed out in reverse CTA order, so a CTA waits only for CTAs the hardware dispatched before it.
// Critical path per block: one 64 x 64 tile update + one 64 x 64 mat-vec + one flag hand-off (~1.5 us), 38 blocks.
// U is the row-major upper triangle (what a column-major LOWER potrf leaves in a row-major buffer): U[i][j] = A[i*lda+j].
#include "common.cuh"

namespace vgg {

namespace {

constexpr int TS_NB = 64;
constexpr int TS_THREADS = 256;
constexpr unsigned long long TS_SENTINEL = 0xffffffffffffffffull;   // x is pre-filled with this NaN pattern

__global__ void __launch_bounds__(TS_THREADS, 1)
    trsv_upper_kernel(int n, int lda, const double* __restrict__ A, const double* __restrict__ y, size_t y_stride,
                      double* __restrict__ x, long long* __restrict__ stamps) {
  extern __shared__ __align__(16) double ts_smem[];
  double(*Ud)[TS_NB + 1] = reinterpret_cast<double(*)[TS_NB + 1]>(ts_smem);                            // diagonal block
  double(*Vi)[TS_NB + 1] = reinterpret_cast<double(*)[TS_NB + 1]>(ts_smem + TS_NB * (TS_NB + 1));      // its inverse
  double* xs = ts_smem + 2 * TS_NB * (TS_NB + 1);
  double* accs = xs + TS_NB;
  const int nb = gridDim.x;
  const int b = nb - 1 - (int)blockIdx.x;     // CTA 0 owns the last block row: a CTA only ever waits for lower-numbered CTAs
  const int r0 = b * TS_NB;
  const int rows = min(TS_NB, n - r0);
  const int tid = threadIdx.x;
  const int r = tid >> 2, seg = tid & 3;      // row of the block, 16-column segment
  // stamps (vgg_dev_trsv_probe only, null in the solve): globaltimer stamps, 6 slots per block row: kernel entry,
  // diagonal block loaded, inverse ready, every x_j consumed, x_b published, right-hand side in place
  auto now_ns = []() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
  };
  if (stamps && tid == 0) stamps[6 * b] = now_ns();
  // this block row's right-hand side, requested FIRST: r02 timestamps showed this one 8-byte load per thread taking
  // ~19 us when it was issued after the inversion (every block row, same absolute completion time) -- and the whole
  // chain waits for the last block row.  Issued here it completes under the block load and the inversion.
  double y_mine = 0.0;
  if (tid < TS_NB && tid < rows) y_mine = __ldcg(&y[(size_t)(r0 + tid) * y_stride]);

  // ---- diagonal block and its inverse (upper triangular; padded rows/cols = identity)
  for (int e = tid; e < TS_NB * TS_NB; e += TS_THREADS) {
    const int i = e / TS_NB, j = e % TS_NB;
    double v = (i == j) ? 1.0 : 0.0;
    if (i < rows && j < rows && j >= i) v = A[(size_t)(r0 + i) * lda + r0 + j];
    Ud[i][j] = v;
  }
  __syncthreads();
  if (stamps && tid == 0) stamps[6 * b + 1] = now_ns();
  if (tid < TS_NB) xs[tid] = 1.0 / Ud[tid][tid];       // reciprocal pivots (xs is free until the first hop)
  __syncthreads();
  {
    // column c = tid / 4 of inv(U) by back substitution U v = e_c (entries below the diagonal are zero); the four threads
    // of a column split every row's dot product over k (one warp holds 8 columns, so a __syncwarp orders the rows).
    // r02 timestamps (tools/microbench.py trsv): with ONE thread per column this start-up took ~50 us of the kernel's
    // 150 -- the chain through the 38 block rows cannot begin before the last block row has its inverse.
    const int c = tid >> 2, part = tid & 3;
    for (int i = TS_NB - 1; i >= 0; --i) {
      double s = 0.0;
      if (i < c) {
        for (int k = i + 1 + part; k <= c; k += 4) s = fma(-Ud[i][k], Vi[k][c], s);
      }
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      if (part == 0) Vi[i][c] = i > c ? 0.0 : (i == c ? xs[i] : s * xs[i]);
      __syncwarp();
    }
  }
  __syncthreads();
  if (stamps && tid == 0) stamps[6 * b + 2] = now_ns();
  // ---- right-hand side rows of this block
  if (tid < TS_NB) accs[tid] = y_mine;
  __syncthreads();
  if (stamps && tid == 0) stamps[6 * b + 5] = now_ns();

  // ---- block columns to the right, last first; tile j+... prefetched into registers before its x is awaited
  // three tiles are kept in flight in registers (tiles do not depend on x, only x_j does)
  double t0[16], t1[16], t2[16];
  auto load_tile = [&](double (&tile)[16], int j) {
    const int c0 = j * TS_NB + seg * 16;
    const double* src = A + (size_t)(r0 + (r < rows ? r : 0)) * lda + c0;
#pragma unroll
    for (int k = 0; k < 16; ++k) tile[k] = (j > b && r < rows && c0 + k < n) ? src[k] : 0.0;
  };
  double acc = 0.0;                            // this thread's partial of row r (its 16-column segment), over all j
  auto hop = [&](const double (&tile)[16], int j) {
    // x_j arrives as data: the buffer was pre-filled with a sentinel NaN pattern, every element is polled by one thread
    // (8-byte stores are single-copy atomic, so no flag, no fence and no second round trip are needed)
    // (r02: one flag per block row watched by one thread per CTA measured 160.6 us against 150.6 us for this hand-off --
    // the fence + flag round trip costs more than the 64-thread polling it removes)
    if (tid < TS_NB) {
      double v = 0.0;
      if (j * TS_NB + tid < n) {
        const volatile unsigned long long* src = reinterpret_cast<const volatile unsigned long long*>(&x[j * TS_NB + tid]);
        unsigned long long bits;
        do {
          bits = *src;
        } while (bits == TS_SENTINEL);
        v = __longlong_as_double((long long)bits);
      }
      xs[tid] = v;
    }
    __syncthreads();
    // four independent chains: the FP64 pipe's dependent-issue latency (~20 cycles) makes one 16-long chain 320 cycles
    // of every hop's critical path
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
    for (int k = 0; k < 16; k += 4) {
      s0 = fma(tile[k], xs[seg * 16 + k], s0);
      s1 = fma(tile[k + 1], xs[seg * 16 + k + 1], s1);
      s2 = fma(tile[k + 2], xs[seg * 16 + k + 2], s2);
      s3 = fma(tile[k + 3], xs[seg * 16 + k + 3], s3);
    }
    acc += (s0 + s1) + (s2 + s3);
    __syncthreads();                           // xs is rewritten in the next round
  };
  int j = nb - 1;
  // The last block row has no block column to its right.  It must not even WALK the (long, straight-line) prefetch and
  // hop code below: r02 timestamps showed it spending 20 us between "inverse ready" and its publication with nothing to
  // compute -- 11 KB of cold instructions fetched line by line -- and every other block row waits for it.
  if (b < nb - 1) {
  load_tile(t0, j);
  load_tile(t1, j - 1);
  load_tile(t2, j - 2);
  while (j > b) {
    hop(t0, j);
    load_tile(t0, j - 3);
    if (--j <= b) break;
    hop(t1, j);
    load_tile(t1, j - 3);
    if (--j <= b) break;
    hop(t2, j);
    load_tile(t2, j - 3);
    --j;
  }
  }
  if (stamps && tid == 0) stamps[6 * b + 3] = now_ns();      // every x_j this block row needs has been consumed
  // reduce the four segments of a row, subtract from the right-hand side
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  if (seg == 0) accs[r] -= acc;
  __syncthreads();
  // ---- x_b = inv(U_bb) acc: four threads per row, published element by element
  {
    double q0 = 0.0, q1 = 0.0, q2 = 0.0, q3 = 0.0;
#pragma unroll
    for (int k = 0; k < 16; k += 4) {
      const int c = seg * 16 + k;
      q0 = fma(c >= r ? Vi[r][c] : 0.0, accs[c], q0);
      q1 = fma(c + 1 >= r ? Vi[r][c + 1] : 0.0, accs[c + 1], q1);
      q2 = fma(c + 2 >= r ? Vi[r][c + 2] : 0.0, accs[c + 2], q2);
      q3 = fma(c + 3 >= r ? Vi[r][c + 3] : 0.0, accs[c + 3], q3);
    }
    double s = (q0 + q1) + (q2 + q3);
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    if (seg == 0 && r < rows) {
      unsigned long long bits = (unsigned long long)__double_as_longlong(s);
      if (s != s) bits = 0x7ff8000000000000ull;        // never publish the sentinel pattern
      *reinterpret_cast<volatile unsigned long long*>(&x[r0 + r]) = bits;
    }
  }
  if (stamps) {
    __syncthreads();
    if (tid == 0) stamps[6 * b + 4] = now_ns();
  }
}

}  // namespace

// x = U^-1 y
int launch_trsv_upper(int n, int lda, const double* A, const double* y, size_t y_stride, double* x, cudaStream_t st) {
  const int nb = (n + TS_NB - 1) / TS_NB;
  VGG_REQUIRE(nb <= 120, "trsv_upper: n too large for one co-resident wave");
  const size_t smem = sizeof(double) * (2 * TS_NB * (TS_NB + 1) + 2 * TS_NB);
  static bool attr = false;
  if (!attr) {
    VGG_CUDA_CHECK(cudaFuncSetAttribute(trsv_upper_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr = true;
  }
  VGG_CUDA_CHECK(cudaMemsetAsync(x, 0xFF, sizeof(double) * (size_t)n, st));   // sentinel fill: x_j is polled as data
  trsv_upper_kernel<<<nb, TS_THREADS, smem, st>>>(n, lda, A, y, y_stride, x, nullptr);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}

}  // namespace vgg

// tools/microbench.py trsv: the backward substitution on a random well-conditioned upper triangle, with per-block-row
// timestamps (ns, globaltimer): stamps_host[2 b] = block row b has consumed every x_j it needs, [2 b + 1] = x_b published
extern "C" int vgg_dev_trsv_probe(int n, int lda, const double* A_dev, const double* y_dev, double* x_dev, long long* stamps_host) {
  using namespace vgg;
  const int nb = (n + TS_NB - 1) / TS_NB;
  static long long* d = nullptr;                      // allocated once: a cudaMalloc / cudaFree pair per call would put
  static int d_cap = 0;                                // allocator work (and its TLB effects) right in front of the kernel
  if (d_cap < 6 * nb) {
    if (d) cudaFree(d);
    VGG_CUDA_CHECK(cudaMalloc(&d, sizeof(long long) * 6 * nb));
    d_cap = 6 * nb;
  }
  VGG_CUDA_CHECK(cudaMemset(d, 0, sizeof(long long) * 6 * nb));
  const size_t smem = sizeof(double) * (2 * TS_NB * (TS_NB + 1) + 2 * TS_NB);
  VGG_CUDA_CHECK(cudaFuncSetAttribute(trsv_upper_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  VGG_CUDA_CHECK(cudaMemset(x_dev, 0xFF, sizeof(double) * (size_t)n));
  trsv_upper_kernel<<<nb, TS_THREADS, smem>>>(n, lda, A_dev, y_dev, 1, x_dev, d);
  VGG_LAUNCH_CHECK();
  VGG_CUDA_CHECK(cudaDeviceSynchronize());
  VGG_CUDA_CHECK(cudaMemcpy(stamps_host, d, sizeof(long long) * 6 * nb, cudaMemcpyDeviceToHost));
  return VGG_OK;
}
