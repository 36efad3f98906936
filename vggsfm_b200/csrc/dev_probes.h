// Development probes (NOT part of the public C ABI in include/vggsfm_b200.h): exported from the library for
// tools/syrk_i8_check.py, tools/microbench.py and bench.py's roofline only.
#pragma once
#ifdef __cplusplus
extern "C" {
#endif
/* Tensor-pipe probe used for the SYRK's roofline: cycles per back-to-back tcgen05.mma.kind::i8 (M=128, K=32); mode
 * bit0 selects N=256 (else 128), mode>>1 the shared-memory layout (0 = 64 B swizzle, 1 = 128 B swizzle, 2 = none).
 * out_cycles is a host pointer. */
int vgg_syrk_ozaki_mma_rate(int iters, int mode, double* out_cycles, void* stream);
/* Kernel-only timing of ba_blocks_kernel: while enabled, every build_blocks call records a CUDA event pair on its stream
 * directly around the kernel launch (the accumulator memsets before it are outside); last_ms waits for the second event
 * and returns the elapsed milliseconds of the most recent launch. */
int vgg_dev_blocks_timing(int enable);
int vgg_dev_blocks_last_ms(double* ms);
/* One-CTA probe of the in-shared-memory POTRF128 of csrc/chol.cu:
 * A_host row-major SPD 128 x 128, L_host its factor, prof13_host[0..5] = cycles per phase seen by warp 0, [6..11] by
 * warp 1 (0 first leaf, 1 TRSM of the micro-panel, 2 look-ahead section work, 3 wait at its barrier, 4 rank-32 DMMA
 * update, 5 first leaf of the next sub-panel), [12] = total cycles of the last of `reps` passes. */
int vgg_dev_chol128_probe(int reps, const double* A_host, double* L_host, long long* prof13_host);
/* Band hint of the tensor-core SYRK for tests: ranges_host[2*rb], [2*rb+1] = the 64-row k-block range outside which the
 * 128-column row block rb of Zt is exactly zero (count = 2 * Dpad/128; count = 0 clears it).  vgg_ba_solve computes the
 * same thing from the visibility mask and clears it when it returns. */
int vgg_dev_set_syrk_ranges(const int* ranges_host, int count);
/* Backward substitution (csrc/trsv.cu) with per-block-row timestamps (ns): stamps_host[2 b] = block row b (64 rows) has
 * consumed every x_j it needs, [2 b + 1] = x_b published.  A_dev: row-major upper triangle, lda columns. */
int vgg_dev_trsv_probe(int n, int lda, const double* A_dev, const double* y_dev, double* x_dev, long long* stamps_host);
/* Block structure for the in-repo Cholesky (tests): end_blk_host[b] = one past the last band block (128 rows) of block
 * column b, arrow_blk = first block of the dense arrow; count = 0 clears it (dense). */
int vgg_dev_set_chol_band(const int* end_blk_host, int count, int arrow_blk);

#ifdef __cplusplus
}
#endif
