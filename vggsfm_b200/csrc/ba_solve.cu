// Levenberg-Marquardt driver (Ceres TrustRegionMinimizer + LevenbergMarquardtStrategy semantics) and
// the C-ABI entry points of the bundle-adjustment path.  The loop body is ~14 kernel launches per
// iteration on one stream and ONE small device->host read (accept/reject scalars); track shards on
// other GPUs join through the caller's all-reduce hook (NCCL over NVLink, see vggsfm_b200/dist.py).
#include <cublas_v2.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <functional>
#include <map>
#include <vector>
#include "common.cuh"

namespace vgg {

static thread_local char g_err[512] = "";
thread_local long long g_launch_count = 0;
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// kernels (ba_blocks.cu / ba_schur.cu)
int ba_build_blocks(const vgg_ba_problem* p, double* cost, double* camrec, double* g_p, double* H_pp, double* W,
                    double* shared_out, int frames_per_cta, cudaStream_t stream, bool outputs_zeroed = false);
int launch_jacobi_scale_points(int N, const double* H_pp, double* sc_p, int enable, cudaStream_t st);
int launch_jacobi_scale_cams(int D, const double* hdiag, double* sc_c, int enable, cudaStream_t st);
int launch_point_prep(int N, const double* H_pp, const double* g_p, const double* sc_p, const uint8_t* point_const,
                      double radius, double min_diag, double max_diag, double* M, double* q, double* dpp,
                      double* scal, cudaStream_t st);
int launch_assemble_hc(int S, int dc, int ns, int KR, int Dpad, const double* camrec, const double* shared_in,
                       double* Sraw, double* rhs, double* hdiag, double* gvec, ptrdiff_t mc_off, cudaStream_t st);
int launch_z_transpose(int D, int N, int Dpad, const double* W, const double* M, const double* q, double* Zt,
                       double* rhs, ptrdiff_t mc_off, cudaStream_t st, unsigned long long* amax);
size_t syrk_i8_workspace_bytes(int Kpad, int Dpad, int slices);
int launch_syrk_i8(int Kpad, int Dpad, const double* Zt, double* Cmat, ptrdiff_t mc_off, int slices, void* ws,
                   size_t ws_bytes, cudaStream_t st, bool amax_ready);
unsigned long long* syrk_i8_amax(void* ws);
int syrk_i8_reset_amax(void* ws, int Dpad, cudaStream_t st);
int launch_scale_damp(int D, int Dpad, double* A, const double* rhs, const double* hdiag, const double* sc,
                      const uint8_t* pconst, double radius, double min_diag, double max_diag, double* bvec,
                      cudaStream_t st);
int launch_cam_step(int D, const double* dcs, size_t dcs_stride, const double* sc, const double* hdiag, const double* gvec,
                    const uint8_t* pconst, double radius, double min_diag, double max_diag, double* d_c, double* scal,
                    cudaStream_t st);
int launch_backsub(int D, int N, const double* W, const double* d_c, double* wacc, cudaStream_t st);
int launch_point_step(int N, const double* M, const double* g_p, const double* wacc, const double* sc_p,
                      const double* dpp, const double* X, double radius, double* Xc, double* scal, cudaStream_t st);
int launch_cam_update(int S, int dc, int ns, int model, const double* d_c, const double* poses, const double* intr,
                      double* poses_c, double* intr_c, cudaStream_t st);
int launch_extract_gvec(int S, int dc, int ns, int KR, const double* camrec, const double* shared_in, double* gvec,
                        cudaStream_t st);
int launch_gradmax(int D, int N, const double* gvec, const uint8_t* pconst, const double* g_p,
                   const uint8_t* point_const, double* scal, cudaStream_t st);

int launch_trsv_upper(int n, int lda, const double* A, const double* y, size_t y_stride, double* x, cudaStream_t st);
size_t chol_workspace_doubles(int n);
int chol_lower_inplace(int n, int lda, double* A, double* Ldiag, int* info, cudaStream_t st);
extern FabricDev g_fabric_dev; // csrc/ba_schur.cu: reduce-scatter destinations read by the SYRK epilogue
int launch_fabric_barrier(const FabricDev& fd, size_t flags_off, unsigned long long epoch, int* err, cudaStream_t st);
int launch_fabric_gather(const FabricDev& fd, int nrows, int nmat, int ncols_vec, int lda, cudaStream_t st);
int launch_fabric_allreduce(const FabricDev& fd, size_t flags_off, size_t mail_off, int mail_len, int parity,
                            unsigned long long epoch, double* vec, int count, int max_slot, int* err, cudaStream_t st);

// gathers the accept/reject scalars into one 24-double record so the host reads them with ONE copy:
// [0..7] = scal[0..7], [8..15] = small[0..7], [16] = factorisation info, [18] = |x|^2, [19] = fabric barrier timeout
__global__ void pack_scalars_kernel(const double* __restrict__ scal, const double* __restrict__ small,
                                    const int* __restrict__ info, double* __restrict__ out) {
  const int i = threadIdx.x;
  if (i < 8) out[i] = scal[i];
  else if (i < 16) out[i] = small[i - 8];
  else if (i == 16) out[i] = (double)info[0];       // chol.cu: non-positive pivot
  else if (i == 18) out[i] = scal[8];              // |x|^2 (xnorm_kernel), 0 unless parameter_tolerance > 0
  else if (i == 19) out[i] = (double)info[2];      // a cross-rank barrier of csrc/fabric.cu timed out
}

// |x|^2 of Ceres' reduced program in ambient coordinates (ParameterToleranceReached: step_norm <= tol * (|x| + tol)):
// unit quaternion + translation of every image whose block is not constant, non-constant camera blocks (f,cx,cy[,k]),
// free points.  Only launched when parameter_tolerance > 0 (COLMAP's BA default is 0).  One CTA; out[0] = |x|^2.
__global__ void xnorm_kernel(int S, int N, int dc, int ns, int model, const uint8_t* __restrict__ pconst,
                             const uint8_t* __restrict__ point_const, const double* __restrict__ poses,
                             const double* __restrict__ intr, const double* __restrict__ pts, double* __restrict__ out) {
  double acc = 0.0;
  const int np = model == VGG_SIMPLE_RADIAL ? 4 : 3;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    const uint8_t* c = pconst + (size_t)s * dc;
    if (!(c[0] && c[1] && c[2])) acc += 1.0;
    if (!(c[3] && c[4] && c[5])) {
      const double* P = poses + (size_t)s * 12;
      acc += P[3] * P[3] + P[7] * P[7] + P[11] * P[11];
    }
    if (dc > 6) {
      bool all_const = true;
      for (int i = 6; i < dc; ++i) all_const = all_const && c[i];
      if (!all_const)
        for (int i = 0; i < np; ++i) acc += intr[(size_t)s * 4 + i] * intr[(size_t)s * 4 + i];
    }
  }
  if (threadIdx.x == 0 && ns > 0) {
    bool all_const = true;
    for (int i = 0; i < ns; ++i) all_const = all_const && pconst[(size_t)S * dc + i];
    if (!all_const)
      for (int i = 0; i < np; ++i) acc += intr[i] * intr[i];
  }
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    if (point_const && point_const[n]) continue;
    acc += pts[3 * (size_t)n] * pts[3 * (size_t)n] + pts[3 * (size_t)n + 1] * pts[3 * (size_t)n + 1] +
           pts[3 * (size_t)n + 2] * pts[3 * (size_t)n + 2];
  }
  __shared__ double red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
    v = warp_sum(v);
    if (threadIdx.x == 0) out[0] = v;
  }
}

// CUDA events of one solve, destroyed on every exit path
struct EventPair {
  cudaEvent_t a = nullptr, b = nullptr;
  ~EventPair() {
    if (a) cudaEventDestroy(a);
    if (b) cudaEventDestroy(b);
  }
};

static double* pinned_scalars() {
  static thread_local double* h = nullptr;
  if (!h) {
    if (cudaHostAlloc(reinterpret_cast<void**>(&h), sizeof(double) * 32, cudaHostAllocDefault) != cudaSuccess) h = nullptr;
  }
  return h;
}

static int dims_of(int model, int mode, int* dc, int* ns, int* KR) {
  if (model != VGG_SIMPLE_PINHOLE && model != VGG_SIMPLE_RADIAL) return VGG_EINVAL;
  const int ni = model == VGG_SIMPLE_PINHOLE ? 1 : 2;
  int d, n;
  if (mode == VGG_INTR_CONST) { d = 6; n = 0; }
  else if (mode == VGG_INTR_PER_FRAME) { d = 6 + ni; n = 0; }
  else if (mode == VGG_INTR_SHARED) { d = 6; n = ni; }
  else return VGG_EINVAL;
  if (dc) *dc = d;
  if (ns) *ns = n;
  if (KR) *KR = d + d * (d + 1) / 2 + 6 * n;
  return VGG_OK;
}

// ------------------------------------------------------------------------------------------------
// workspace layout
// ------------------------------------------------------------------------------------------------
struct BlockSet {
  double *cost, *camrec, *g_p, *H_pp, *W, *shared;
};
struct Layout {
  int S, N, dc, ns, KR, D, Dpad, Kpad;
  BlockSet blk[2];
  double *poses[2], *intr[2], *points[2];
  double *sc_c, *sc_p, *M, *q, *dpp, *wacc, *d_c, *bvec, *Zt;
  double *AR;        // [D*Dpad | rhs Dpad | hdiag Dpad | gvec Dpad]  (one all-reduce)
  double *small;     // [8 scalars | gvec_candidate Dpad]           (one small all-reduce)
  double *scal;      // [16]
  double *packed;    // [24] scalars gathered for the host
  double *chol_diag;
  int *dev_info;
  uint8_t* oz_ws;    // int8 slices + scales of the tensor-core SYRK (csrc/syrk_i8.cu)
  size_t oz_bytes;
  size_t bytes;
};

// The Schur SYRK runs on the tensor cores (tcgen05 INT8 Ozaki slices, csrc/syrk_i8.cu) with 7 slices = 54 fractional
// bits, FP64-equivalent.  It replaced the FP64-pipe DMMA / DFMA kernels: 2.46 ms -> 1.10 ms per iteration at C3 on a
// B200, same iterates (profiles/r01_*).
constexpr int kSyrkSlices = 7;

static int make_layout(int S, int N, int model, int mode, void* base, size_t cap, Layout* L) {
  int dc, ns, KR;
  if (dims_of(model, mode, &dc, &ns, &KR) != VGG_OK) {
    set_error("bad camera_model/intr_mode");
    return VGG_EINVAL;
  }
  L->S = S; L->N = N; L->dc = dc; L->ns = ns; L->KR = KR;
  L->D = S * dc + ns;
  L->Dpad = (int)align_up((size_t)L->D + 2, 128);      // >= 2 spare slots after D (fabric-mode scalar sync)
  L->Kpad = (int)align_up((size_t)3 * N, 16);
  Carver c(base, cap);
  for (int b = 0; b < 2; ++b) {
    L->blk[b].cost = c.take<double>(8);
    L->blk[b].shared = c.take<double>(8);
    L->blk[b].camrec = c.take<double>((size_t)S * KR);
    L->blk[b].g_p = c.take<double>((size_t)N * 3);
    L->blk[b].H_pp = c.take<double>((size_t)N * 6);
    L->blk[b].W = c.take<double>((size_t)(L->D + (L->D & 1)) * N * 3);   // track-major [N][pitch][3]
    L->poses[b] = c.take<double>((size_t)S * 12);
    L->intr[b] = c.take<double>((size_t)S * 4);
    L->points[b] = c.take<double>((size_t)N * 3);
  }
  L->sc_c = c.take<double>(L->Dpad);
  L->sc_p = c.take<double>((size_t)N * 3);
  L->M = c.take<double>((size_t)N * 9);
  L->q = c.take<double>((size_t)N * 3);
  L->dpp = c.take<double>((size_t)N * 3);
  L->wacc = c.take<double>((size_t)N * 3);
  L->d_c = c.take<double>(L->Dpad);
  L->bvec = c.take<double>(L->Dpad);
  L->Zt = c.take<double>((size_t)L->Kpad * L->Dpad);
  L->AR = c.take<double>((size_t)L->D * L->Dpad + 3 * (size_t)L->Dpad);
  L->small = c.take<double>(8 + (size_t)L->Dpad);
  L->scal = c.take<double>(16);
  L->packed = c.take<double>(32);
  L->chol_diag = c.take<double>(chol_workspace_doubles(L->D + 1));
  L->dev_info = c.take<int>(4);
  L->oz_bytes = syrk_i8_workspace_bytes(L->Kpad, L->Dpad, kSyrkSlices);
  c.off = align_up(c.off, 1024);
  L->oz_ws = c.take<uint8_t>(L->oz_bytes);
  L->bytes = align_up(c.off, 256);
  if (base && c.off > cap) {
    set_error("workspace too small: need %zu bytes, have %zu", c.off, cap);
    return VGG_EWORKSPACE;
  }
  return VGG_OK;
}

static cublasHandle_t get_cublas() {
  static thread_local cublasHandle_t h = nullptr;
  if (!h) {
    if (cublasCreate(&h) != CUBLAS_STATUS_SUCCESS) h = nullptr;
  }
  return h;
}

// Layout of the symmetric allocation of fabric v2 (doubles): two copies of the reduced system (iteration parity, so a
// rank may zero the next copy while a slow peer still pulls from the previous one), the mailboxes of the small
// all-reduce (2 parities x 8 source ranks), one row of 64-bit barrier flags.
struct FabricLayout {
  size_t arc, mail_off, flags_off, total;
  int mail_len;
};
static FabricLayout fabric_layout(int D, int Dpad) {
  FabricLayout f;
  f.arc = align_up((size_t)D * Dpad + 3 * (size_t)Dpad, 256);
  f.mail_len = Dpad + 64;
  f.mail_off = 2 * f.arc;
  f.flags_off = align_up(f.mail_off + (size_t)2 * 8 * f.mail_len, 32);
  f.total = f.flags_off + 64;
  return f;
}

// Run-time state of fabric v2 (csrc/fabric.cu): reduce-scatter + gather of the reduced system, in-kernel barriers and
// small all-reduces -- no NCCL call and no host callback inside the LM loop.
struct Fabric2 {
  bool on = false;
  FabricDev base{};                 // peer[r] = base of rank r's symmetric allocation
  FabricLayout lay{};
  unsigned long long* epoch = nullptr;
  int small_parity = 0;
  int* err = nullptr;
  FabricDev at(size_t off) const {
    FabricDev f = base;
    for (int r = 0; r < f.world; ++r) f.peer[r] += off;
    return f;
  }
  int barrier(cudaStream_t st) { return launch_fabric_barrier(base, lay.flags_off, ++*epoch, err, st); }
  int allreduce(double* vec, int count, int max_slot, cudaStream_t st) {
    small_parity ^= 1;
    return launch_fabric_allreduce(base, lay.flags_off, lay.mail_off, lay.mail_len, small_parity, ++*epoch, vec, count,
                                   max_slot, err, st);
  }
};

extern std::vector<int> g_syrk_kb_ranges;     // csrc/syrk_i8.cu: band hint of the current solve
extern std::vector<int> g_chol_band_end;      // csrc/chol.cu: block structure of the reduced system (banded + arrow)
extern int g_chol_arrow_blk;
extern BandDev g_band_dev;                    // csrc/ba_schur.cu: device tables for ba_blocks / z_build / backsub

// resets the process-wide kernel switches when a solve ends, on every exit path
struct SolveGuard {
  ~SolveGuard() {
    g_fabric_dev.world = 0;
    g_syrk_kb_ranges.clear();
    g_chol_band_end.clear();
    g_chol_arrow_blk = 0;
    g_band_dev = BandDev{nullptr, nullptr, nullptr, 0};
  }
};

// first / last visible point of every frame (N / -1 when the frame sees nothing): the band structure of sequential
// (video) problems, where a point lives for a few windows and the dense [S, N] grid is mostly masked out
__global__ void __launch_bounds__(256) frame_point_range_kernel(int S, int N, const uint8_t* __restrict__ mask,
                                                                int* __restrict__ out) {
  __shared__ int s_lo[256], s_hi[256];
  const int s = blockIdx.x;
  int lo = N, hi = -1;
  for (int n = threadIdx.x; n < N; n += 256)
    if (mask[(size_t)s * N + n]) {
      lo = min(lo, n);
      hi = max(hi, n);
    }
  s_lo[threadIdx.x] = lo;
  s_hi[threadIdx.x] = hi;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) {
      s_lo[threadIdx.x] = min(s_lo[threadIdx.x], s_lo[threadIdx.x + w]);
      s_hi[threadIdx.x] = max(s_hi[threadIdx.x], s_hi[threadIdx.x + w]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[2 * s] = s_lo[0];
    out[2 * s + 1] = s_hi[0];
  }
}

// Per 128-column row block of Zt: the 64-row k-block range outside which the block is exactly zero (Zt row 3n+c belongs to
// point n; column d < S*dc to frame d / dc; the shared-intrinsics columns see every point).  Leaves the hint empty when
// the grid is (nearly) dense.  One small kernel + a 8 S byte read-back per solve.
static int compute_band_hint(const vgg_ba_problem* prob, int dc, int D, int Dpad, int Kpad, bool multi_rank, cudaStream_t st) {
  g_syrk_kb_ranges.clear();
  g_chol_band_end.clear();
  g_chol_arrow_blk = 0;
  g_band_dev = BandDev{nullptr, nullptr, nullptr, 0};
  const char* env = getenv("VGG_BAND");                 // read per solve so that a test can compare both paths in one process
  const bool off = env && env[0] == '0';
  const int S = prob->S, N = prob->N, nb = Dpad / 128, KB = (Kpad + 63) / 64;
  if (off || nb < 6 || N < 1024) return VGG_OK;
  static thread_local int* dev = nullptr;
  static thread_local int cap = 0;
  if (cap < 2 * S) {
    if (dev) cudaFree(dev);
    VGG_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&dev), sizeof(int) * 2 * (size_t)S));
    cap = 2 * S;
  }
  frame_point_range_kernel<<<S, 256, 0, st>>>(S, N, prob->mask, dev);
  VGG_LAUNCH_CHECK();
  std::vector<int> fr(2 * (size_t)S);
  VGG_CUDA_CHECK(cudaMemcpyAsync(fr.data(), dev, sizeof(int) * fr.size(), cudaMemcpyDeviceToHost, st));
  VGG_CUDA_CHECK(cudaStreamSynchronize(st));
  std::vector<int> rg(2 * (size_t)nb);
  for (int rb = 0; rb < nb; ++rb) {
    const int d0 = rb * 128, d1 = std::min(D, d0 + 128) - 1;
    int lo = KB, hi = 0;
    if (d1 >= d0) {
      if (d1 >= S * dc) {
        lo = 0;
        hi = KB;
      } else {
        for (int f = d0 / dc; f <= d1 / dc; ++f) {
          if (fr[2 * f + 1] < 0) continue;
          lo = std::min(lo, 3 * fr[2 * f] / 64);
          hi = std::max(hi, (3 * fr[2 * f + 1] + 2) / 64 + 1);
        }
      }
    }
    if (hi <= lo) lo = hi = 0;
    rg[2 * rb] = lo;
    rg[2 * rb + 1] = std::min(hi, KB);
  }
  // worth it only if a good part of the tile x k volume disappears
  double kept = 0.0, all = 0.0;
  for (int bi = 0; bi < nb; ++bi)
    for (int bj = 0; bj <= bi; ++bj) {
      all += KB;
      kept += std::max(0, std::min(rg[2 * bi + 1], rg[2 * bj + 1]) - std::max(rg[2 * bi], rg[2 * bj]));
    }
  if (kept < 0.7 * all) {
    g_syrk_kb_ranges = rg;
    // the same structure for the factorisation: block (i, b) of the reduced system is non-zero iff the k ranges of row
    // blocks i and b meet; the blocks from the first shared-intrinsics column on (and the bordered right-hand-side row)
    // are the dense "arrow".  end[b] = one past the last band block of column b, made non-decreasing (the envelope
    // Cholesky fills) and >= b + 2 so that block row b + 1 always counts as band.
    // Multi-GPU solves: the ranges above describe THIS rank's tracks only, which is all the kernels that touch its W / Zt
    // need; the reduced system it factors is the sum over ranks, so the factorisation keeps the dense structure there.
    const int arrow = (S * dc) / 128;
    if (arrow >= 4 && !multi_rank) {
      std::vector<int> end(nb);
      int prev = 0;
      for (int b = 0; b < nb; ++b) {
        int e = b;
        if (b < arrow) {
          for (int i = b + 1; i < arrow; ++i)
            if (std::min(rg[2 * i + 1], rg[2 * b + 1]) > std::max(rg[2 * i], rg[2 * b])) e = i;
          e = std::max(e + 1, std::min(b + 2, arrow));
          e = std::max(e, prev);
          e = std::min(e, arrow);
        } else {
          e = nb;
        }
        end[b] = e;
        prev = e;
      }
      g_chol_band_end = end;
      g_chol_arrow_blk = arrow;
      // device tables for the kernels that walk the dense [frames, points] grid (VGG_BAND=2: SYRK/Cholesky hint only)
      if (!(env && env[0] == '2')) {
        const int ngroups = (S + 31) / 32;
        std::vector<int> tab(2 * (size_t)(nb + KB + ngroups), 0);
        int* t_rb = tab.data();
        int* t_kb = t_rb + 2 * nb;
        int* t_fg = t_kb + 2 * KB;
        for (int i = 0; i < 2 * nb; ++i) t_rb[i] = rg[i];
        for (int kb = 0; kb < KB; ++kb) {
          int first = -1, last = -1;
          for (int rb = 0; rb < arrow; ++rb)
            if (rg[2 * rb] <= kb && kb < rg[2 * rb + 1]) {
              if (first < 0) first = rb;
              last = rb;
            }
          t_kb[2 * kb] = first < 0 ? 0 : first * 128;
          t_kb[2 * kb + 1] = first < 0 ? 0 : (last + 1) * 128;
        }
        for (int g = 0; g < ngroups; ++g) {
          int lo = N, hi = 0;
          for (int f = 32 * g; f < std::min(S, 32 * g + 32); ++f) {
            if (fr[2 * f + 1] < 0) continue;
            lo = std::min(lo, fr[2 * f]);
            hi = std::max(hi, fr[2 * f + 1] + 1);
          }
          t_fg[2 * g] = hi > lo ? lo : 0;
          t_fg[2 * g + 1] = hi > lo ? hi : 0;
        }
        static thread_local int* tdev = nullptr;
        static thread_local size_t tcap = 0;
        if (tcap < tab.size()) {
          if (tdev) cudaFree(tdev);
          VGG_CUDA_CHECK(cudaMalloc(reinterpret_cast<void**>(&tdev), sizeof(int) * tab.size()));
          tcap = tab.size();
        }
        VGG_CUDA_CHECK(cudaMemcpyAsync(tdev, tab.data(), sizeof(int) * tab.size(), cudaMemcpyHostToDevice, st));
        VGG_CUDA_CHECK(cudaStreamSynchronize(st));           // pageable source
        g_band_dev = BandDev{tdev, tdev + 2 * nb, tdev + 2 * (nb + KB), arrow * 128};
      }
    }
  }
  return VGG_OK;
}

// Schur complement of blk onto AR (Sraw, rhs, hdiag, gvec) at the given radius
static int schur_build(const Layout& L, const BlockSet& b, const uint8_t* point_const, double radius, double min_diag,
                       double max_diag, cudaStream_t st, ptrdiff_t mc_off = 0,
                       const std::function<int()>* barrier = nullptr) {
  int rc;
  double* Sraw = L.AR;
  double* rhs = L.AR + (size_t)L.D * L.Dpad;
  double* hdiag = rhs + L.Dpad;
  double* gvec = hdiag + L.Dpad;
  if ((rc = launch_point_prep(L.N, b.H_pp, b.g_p, L.sc_p, point_const, radius, min_diag, max_diag, L.M, L.q, L.dpp,
                              L.scal, st)))
    return rc;
  VGG_CUDA_CHECK(cudaMemsetAsync(L.AR, 0, sizeof(double) * ((size_t)L.D * L.Dpad + 3 * (size_t)L.Dpad), st));
  // fabric mode: every rank's copy must be zero before anyone's multimem reductions land in it
  if (mc_off && barrier && (rc = (*barrier)())) return rc;
  if ((rc = launch_assemble_hc(L.S, L.dc, L.ns, L.KR, L.Dpad, b.camrec, b.shared, Sraw, rhs, hdiag, gvec, mc_off, st))) return rc;
  if ((rc = syrk_i8_reset_amax(L.oz_ws, L.Dpad, st))) return rc;
  if ((rc = launch_z_transpose(L.D, L.N, L.Dpad, b.W, L.M, L.q, L.Zt, rhs, mc_off, st, syrk_i8_amax(L.oz_ws)))) return rc;
  if ((rc = launch_syrk_i8(L.Kpad, L.Dpad, L.Zt, Sraw, mc_off, kSyrkSlices, L.oz_ws, L.oz_bytes, st, true))) return rc;
  // ... and all reductions must have landed before anyone reads its copy
  if (mc_off && barrier && (rc = (*barrier)())) return rc;
  return VGG_OK;
}

}  // namespace vgg

using namespace vgg;

extern "C" {

const char* vgg_last_error(void) { return g_err; }
int vgg_version(void) { return 100; }

void vgg_ba_default_options(vgg_ba_options* o) {
  memset(o, 0, sizeof(*o));
  o->max_num_iterations = 100;
  o->max_num_consecutive_invalid_steps = 10;
  o->jacobi_scaling = 1;
  o->function_tolerance = 0.0;
  o->gradient_tolerance = 1e-4;
  o->parameter_tolerance = 0.0;
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
}

int vgg_ba_dims(int camera_model, int intr_mode, int* dc, int* ns) {
  return dims_of(camera_model, intr_mode, dc, ns, nullptr);
}

int vgg_ba_camrec_len(int camera_model, int intr_mode) {
  int KR = 0;
  if (dims_of(camera_model, intr_mode, nullptr, nullptr, &KR) != VGG_OK) return VGG_EINVAL;
  return KR;
}

int vgg_ba_workspace_bytes(int S, int N, int camera_model, int intr_mode, size_t* bytes) {
  VGG_REQUIRE(S > 0 && N > 0 && bytes, "S, N must be positive");
  int dc, ns;
  if (dims_of(camera_model, intr_mode, &dc, &ns, nullptr) != VGG_OK) {
    set_error("bad camera_model/intr_mode");
    return VGG_EINVAL;
  }
  Layout L;
  const int rc = make_layout(S, N, camera_model, intr_mode, nullptr, 0, &L);
  if (rc) return rc;
  *bytes = L.bytes;
  return VGG_OK;
}

int vgg_ba_build_blocks(const vgg_ba_problem* prob, double* cost, double* camrec, double* g_p, double* H_pp, double* W,
                        double* shared_out, int frames_per_cta, void* stream) {
  VGG_REQUIRE(prob && cost && camrec && g_p && H_pp && W && shared_out, "null pointer");
  g_launch_count = 0;
  return ba_build_blocks(prob, cost, camrec, g_p, H_pp, W, shared_out, frames_per_cta, (cudaStream_t)stream);
}

int vgg_ba_schur(const vgg_ba_problem* prob, const double* camrec, const double* g_p, const double* H_pp,
                 const double* W, const double* shared_in, const double* scale_p, double radius, double min_diag,
                 double max_diag, void* workspace, size_t ws_bytes, double* Sraw, double* rhs, int* Dpad_out,
                 void* stream) {
  VGG_REQUIRE(prob && workspace && Sraw && rhs, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  g_launch_count = 0;
  Layout L;
  int rc = make_layout(prob->S, prob->N, prob->camera_model, prob->intr_mode, workspace, ws_bytes, &L);
  if (rc) return rc;
  BlockSet b;
  b.cost = nullptr;
  b.camrec = const_cast<double*>(camrec);
  b.g_p = const_cast<double*>(g_p);
  b.H_pp = const_cast<double*>(H_pp);
  b.W = const_cast<double*>(W);
  b.shared = const_cast<double*>(shared_in);
  VGG_CUDA_CHECK(cudaMemcpyAsync(L.sc_p, scale_p, sizeof(double) * (size_t)L.N * 3, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemsetAsync(L.Zt, 0, sizeof(double) * (size_t)L.Kpad * L.Dpad, st));
  VGG_CUDA_CHECK(cudaMemsetAsync(L.scal, 0, sizeof(double) * 16, st));
  rc = schur_build(L, b, prob->point_const, radius, min_diag, max_diag, st);
  if (rc) return rc;
  VGG_CUDA_CHECK(cudaMemcpyAsync(Sraw, L.AR, sizeof(double) * (size_t)L.D * L.Dpad, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemcpyAsync(rhs, L.AR + (size_t)L.D * L.Dpad, sizeof(double) * L.Dpad, cudaMemcpyDeviceToDevice, st));
  if (Dpad_out) *Dpad_out = L.Dpad;
  return VGG_OK;
}

int vgg_cholesky_lower(int n, int lda, double* A, void* workspace, size_t ws_bytes, int* info_host, void* stream) {
  VGG_REQUIRE(A && workspace && n > 0 && lda >= n, "bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  g_launch_count = 0;
  const size_t need = sizeof(double) * chol_workspace_doubles(n) + 256;
  if (ws_bytes < need) {
    set_error("cholesky workspace too small: need %zu bytes", need);
    return VGG_EWORKSPACE;
  }
  int* info = reinterpret_cast<int*>(workspace);
  double* diag = reinterpret_cast<double*>(reinterpret_cast<char*>(workspace) + 256);
  int rc = chol_lower_inplace(n, lda, A, diag, info, st);
  if (rc) return rc;
  if (info_host) {
    VGG_CUDA_CHECK(cudaMemcpyAsync(info_host, info, sizeof(int), cudaMemcpyDeviceToHost, st));
    VGG_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  return VGG_OK;
}

int vgg_ba_reduced_system_doubles(int S, int camera_model, int intr_mode, size_t* doubles) {
  int dc, ns;
  if (!doubles || dims_of(camera_model, intr_mode, &dc, &ns, nullptr) != VGG_OK) {
    set_error("bad camera_model/intr_mode");
    return VGG_EINVAL;
  }
  const size_t D = (size_t)S * dc + ns, Dpad = align_up(D + 2, 128);
  *doubles = D * Dpad + 3 * Dpad;
  return VGG_OK;
}

int vgg_ba_fabric_doubles(int S, int camera_model, int intr_mode, size_t* doubles) {
  int dc, ns;
  if (!doubles || dims_of(camera_model, intr_mode, &dc, &ns, nullptr) != VGG_OK) {
    set_error("bad camera_model/intr_mode");
    return VGG_EINVAL;
  }
  const int D = S * dc + ns;
  *doubles = fabric_layout(D, (int)align_up((size_t)D + 2, 128)).total;
  return VGG_OK;
}

int vgg_ba_solve(const vgg_ba_problem* prob, const vgg_ba_options* opt_in, void* workspace, size_t ws_bytes,
                 vgg_allreduce_fn allreduce, void* ar_user, vgg_ba_summary* summary, double* trace, void* stream) {
  return vgg_ba_solve_fabric(prob, opt_in, workspace, ws_bytes, allreduce, ar_user, nullptr, summary, trace, stream);
}

int vgg_ba_solve_fabric(const vgg_ba_problem* prob, const vgg_ba_options* opt_in, void* workspace, size_t ws_bytes,
                        vgg_allreduce_fn allreduce, void* ar_user, const vgg_ba_fabric* fabric, vgg_ba_summary* summary,
                        double* trace, void* stream) {
  VGG_REQUIRE(prob && workspace && summary, "null pointer");
  VGG_REQUIRE(prob->uv && prob->mask && prob->param_const && prob->poses && prob->intr && prob->points, "null problem array");
  cudaStream_t st = (cudaStream_t)stream;
  g_launch_count = 0;
  vgg_ba_options opt;
  if (opt_in) opt = *opt_in;
  else vgg_ba_default_options(&opt);
  const int S = prob->S, N = prob->N;
  int dc, ns;
  if (dims_of(prob->camera_model, prob->intr_mode, &dc, &ns, nullptr) != VGG_OK) {
    set_error("bad camera_model/intr_mode");
    return VGG_EINVAL;
  }
  const int D = S * dc + ns;
  Layout L;
  int rc = make_layout(S, N, prob->camera_model, prob->intr_mode, workspace, ws_bytes, &L);
  if (rc) return rc;
  const size_t ar_count = (size_t)D * L.Dpad + 3 * (size_t)L.Dpad;
  // fabric mode: the reduced system lives in symmetric (peer-mapped) memory and is reduced by multimem operations
  // issued from the producing kernels; mc_off is the distance from a local address to its multicast twin
  ptrdiff_t mc_off = 0;
  Fabric2 fab2;
  SolveGuard guard;
  static thread_local std::map<const double*, unsigned long long> fabric_epochs;
  if (fabric && fabric->ar_local && fabric->ar_multicast) {
    VGG_REQUIRE(fabric->ar_doubles >= ar_count, "fabric buffer too small (vgg_ba_reduced_system_doubles)");
    L.AR = fabric->ar_local;
    mc_off = fabric->ar_multicast - fabric->ar_local;
    // v2 (default when the caller passed the peer table): VGG_FABRIC=1 keeps v1 (multimem all-reduce into every copy,
    // barriers and small all-reduces through the host hook) for A/B
    static const bool want_v2 = [] { const char* e = getenv("VGG_FABRIC"); return !(e && e[0] == '1'); }();
    const FabricLayout lay = fabric_layout(D, L.Dpad);
    if (want_v2 && fabric->world > 1 && fabric->world <= 8 && fabric->peer_base[0] && fabric->total_doubles >= lay.total) {
      fab2.on = true;
      fab2.lay = lay;
      fab2.base.world = fabric->world;
      fab2.base.rank = fabric->rank;
      for (int r = 0; r < fabric->world; ++r) fab2.base.peer[r] = fabric->peer_base[r];
      fab2.epoch = &fabric_epochs[fabric->peer_base[fabric->rank]];
      fab2.err = L.dev_info + 2;
    } else {
      VGG_REQUIRE(allreduce, "fabric v1 needs the hook for its barrier (op 2)");
    }
  }
  if ((rc = compute_band_hint(prob, dc, D, L.Dpad, L.Kpad, allreduce != nullptr || fabric != nullptr, st))) return rc;
  if (g_band_dev.fg_tracks) {
    // the kernels skip the (track chunk, frame group) regions no observation falls into: their W blocks must read as zero
    const size_t w_doubles = (size_t)N * (size_t)(D + (D & 1)) * 3;
    VGG_CUDA_CHECK(cudaMemsetAsync(L.blk[0].W, 0, sizeof(double) * w_doubles, st));
    VGG_CUDA_CHECK(cudaMemsetAsync(L.blk[1].W, 0, sizeof(double) * w_doubles, st));
  }
  double* Sraw = L.AR;
  double* rhs = L.AR + (size_t)D * L.Dpad;
  double* hdiag = rhs + L.Dpad;
  double* gvec = hdiag + L.Dpad;
  const std::function<int()> barrier_fn = [&]() -> int {
    if (fab2.on) return fab2.barrier(st);
    return allreduce(ar_user, nullptr, 0, 2, st);
  };
  // sum (and one max slot) of a small vector over the ranks: in-kernel over the fabric, else through the host hook
  auto reduce_small = [&](double* vec, size_t count, int op) -> int {
    if (fab2.on) return fab2.allreduce(vec, (int)count, op == 1 ? 0 : -1, st);
    if (allreduce) return allreduce(ar_user, vec, count, op, st);
    return VGG_OK;
  };
  EventPair evs;
  VGG_CUDA_CHECK(cudaEventCreate(&evs.a));
  VGG_CUDA_CHECK(cudaEventCreate(&evs.b));
  const cudaEvent_t ev0 = evs.a, ev1 = evs.b;
  VGG_CUDA_CHECK(cudaEventRecord(ev0, st));

  int cur = 0;
  VGG_CUDA_CHECK(cudaMemcpyAsync(L.poses[0], prob->poses, sizeof(double) * (size_t)S * 12, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemcpyAsync(L.intr[0], prob->intr, sizeof(double) * (size_t)S * 4, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemcpyAsync(L.points[0], prob->points, sizeof(double) * (size_t)N * 3, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemsetAsync(L.Zt, 0, sizeof(double) * (size_t)L.Kpad * L.Dpad, st));
  VGG_CUDA_CHECK(cudaMemsetAsync(L.d_c, 0, sizeof(double) * L.Dpad, st));

  auto eval = [&](int which) -> int {
    vgg_ba_problem p = *prob;
    p.poses = L.poses[which];
    p.intr = L.intr[which];
    p.points = L.points[which];
    const BlockSet& b = L.blk[which];
    // cost | shared | camrec | g_p | H_pp are carved back to back: one memset covers all accumulators
    const size_t acc_bytes = reinterpret_cast<char*>(b.H_pp + (size_t)N * 6) - reinterpret_cast<char*>(b.cost);
    VGG_CUDA_CHECK(cudaMemsetAsync(b.cost, 0, acc_bytes, st));
    return ba_build_blocks(&p, b.cost, b.camrec, b.g_p, b.H_pp, b.W, b.shared, 0, st, true);
  };
  // global cost + gradient max-norm of block set `which`; result lands in host h[0..2] = cost, gmax_c, gmax_p
  double* h_scal = pinned_scalars();
  if (!h_scal) {
    set_error("cudaHostAlloc for the scalar read-back failed");
    return VGG_ECUDA;
  }
  VGG_CUDA_CHECK(cudaMemsetAsync(L.dev_info, 0, sizeof(int) * 4, st));
  auto read_scalars = [&]() -> int {
    pack_scalars_kernel<<<1, 32, 0, st>>>(L.scal, L.small, L.dev_info, L.packed);
    VGG_LAUNCH_CHECK();
    VGG_CUDA_CHECK(cudaMemcpyAsync(h_scal, L.packed, sizeof(double) * 24, cudaMemcpyDeviceToHost, st));   // [0..19] used
    VGG_CUDA_CHECK(cudaStreamSynchronize(st));
    return VGG_OK;
  };
  auto cost_and_gradient = [&](int which, double* cost_out, double* gmax_out) -> int {
    const BlockSet& b = L.blk[which];
    int r;
    VGG_CUDA_CHECK(cudaMemsetAsync(L.small, 0, sizeof(double) * (8 + (size_t)L.Dpad), st));
    VGG_CUDA_CHECK(cudaMemcpyAsync(L.small, b.cost, sizeof(double), cudaMemcpyDeviceToDevice, st));
    if ((r = launch_extract_gvec(S, dc, ns, L.KR, b.camrec, b.shared, L.small + 8, st))) return r;
    if ((r = reduce_small(L.small, 8 + (size_t)L.Dpad, 0))) return r;
    VGG_CUDA_CHECK(cudaMemsetAsync(L.scal + 4, 0, sizeof(double) * 2, st));
    if ((r = launch_gradmax(D, N, L.small + 8, prob->param_const, b.g_p, prob->point_const, L.scal, st))) return r;
    if ((r = reduce_small(L.scal + 5, 1, 1))) return r;
    if ((r = read_scalars())) return r;
    if (h_scal[19] != 0.0) {
      set_error("fabric barrier timed out: a peer rank did not arrive");
      return VGG_ECUDA;
    }
    *cost_out = h_scal[8];
    *gmax_out = fmax(h_scal[4], h_scal[5]);
    return VGG_OK;
  };

  if ((rc = eval(cur))) return rc;
  if ((rc = launch_jacobi_scale_points(N, L.blk[cur].H_pp, L.sc_p, opt.jacobi_scaling, st))) return rc;
  double cost = 0, gmax = 0;
  if ((rc = cost_and_gradient(cur, &cost, &gmax))) return rc;

  memset(summary, 0, sizeof(*summary));
  summary->initial_cost = cost;
  summary->termination = VGG_BA_NO_CONVERGENCE;
  double radius = opt.initial_trust_region_radius;
  double decrease_factor = 2.0;
  int it = 0, invalid_steps = 0;
  bool have_scale_c = false;
  bool done = gmax <= opt.gradient_tolerance;
  if (done) summary->termination = VGG_BA_CONVERGENCE_GRADIENT;

  while (!done) {
    if (it >= opt.max_num_iterations) break;
    if (radius < opt.min_trust_region_radius) {
      summary->termination = VGG_BA_MIN_TRUST_REGION;
      break;
    }
    ++it;
    const int cand = cur ^ 1;
    VGG_CUDA_CHECK(cudaMemsetAsync(L.scal, 0, sizeof(double) * 16, st));
    if (fab2.on) {
      // this iteration's copy of the reduced system (parity) and where the SYRK epilogue sends each row block
      const size_t off = (size_t)(it & 1) * fab2.lay.arc;
      L.AR = fabric->ar_local + off;
      Sraw = L.AR;
      rhs = L.AR + (size_t)D * L.Dpad;
      hdiag = rhs + L.Dpad;
      gvec = hdiag + L.Dpad;
      g_fabric_dev = fab2.at(off);
    }
    if ((rc = schur_build(L, L.blk[cur], prob->point_const, radius, opt.min_lm_diagonal, opt.max_lm_diagonal, st, mc_off,
                          (fab2.on || allreduce) ? &barrier_fn : nullptr)))
      return rc;
    if (fab2.on) {
      // every row block is complete on its owner: pull the others (matrix rows 0..D incl. the rhs row, then hdiag, gvec)
      if ((rc = launch_fabric_gather(g_fabric_dev, D + 3, D + 1, D, L.Dpad, st))) return rc;
      g_fabric_dev.world = 0;
    }
    if (allreduce && !mc_off && (rc = allreduce(ar_user, L.AR, ar_count, 0, st))) return rc;
    if (!have_scale_c) {
      if ((rc = launch_jacobi_scale_cams(D, hdiag, L.sc_c, opt.jacobi_scaling, st))) return rc;
      have_scale_c = true;
    }
    if ((rc = launch_scale_damp(D, L.Dpad, Sraw, rhs, hdiag, L.sc_c, prob->param_const, radius, opt.min_lm_diagonal,
                                opt.max_lm_diagonal, L.bvec, st)))
      return rc;
    // Factor the reduced system: the in-repo blocked Cholesky (csrc/chol.cu) on the row-major LOWER triangle of the
    // BORDERED matrix of order D+1 -- scale_damp put the scaled right-hand side into row D, so the factorisation leaves
    // y = L^-1 b there (and, mirrored like every panel, in column D): the forward substitution costs nothing and only the
    // backward substitution L^T x = y remains.  It replaced cuSOLVER potrf (1.145 ms vs 0.88 ms at n = 2403 on a B200,
    // profiles/r02_*).
    if ((rc = chol_lower_inplace(D + 1, L.Dpad, Sraw, L.chol_diag, L.dev_info, st))) return rc;
    // Backward substitution on U = L^T (the row-major upper triangle), y = column D of the buffer.
    const double* dcs = L.bvec;
    size_t dcs_stride = 1;
    if (D > 7000) {                                   // own kernel needs one co-resident wave of D/64 CTAs
      cublasHandle_t cb = get_cublas();
      if (!cb || cublasSetStream(cb, st) != CUBLAS_STATUS_SUCCESS) {
        set_error("cublasCreate / cublasSetStream failed");
        return VGG_ESOLVER;
      }
      if (cublasDtrsv(cb, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_T, CUBLAS_DIAG_NON_UNIT, D, Sraw, L.Dpad, Sraw + D, L.Dpad) !=
          CUBLAS_STATUS_SUCCESS) {
        set_error("cublasDtrsv failed to launch");
        return VGG_ESOLVER;
      }
      g_launch_count += 1;
      dcs = Sraw + D;
      dcs_stride = (size_t)L.Dpad;
    } else {
      // own backward substitution (csrc/trsv.cu): one launch, block rows chained through the solution vector
      if ((rc = launch_trsv_upper(D, L.Dpad, Sraw, Sraw + D, (size_t)L.Dpad, L.bvec, st))) return rc;
    }
    if ((rc = launch_cam_step(D, dcs, dcs_stride, L.sc_c, hdiag, gvec, prob->param_const, radius, opt.min_lm_diagonal,
                              opt.max_lm_diagonal, L.d_c, L.scal, st)))
      return rc;
    if (mc_off && !fab2.on) {
      // Fabric v1: the multimem reductions reach each rank's copy in a different order, so the copies (and with
      // them the factorisation and the camera step) differ in the last bits.  Keep the replicated camera state
      // and the accept/reject scalars bit-identical on every rank: element-wise MAX over ranks of
      // [d_c | quad_c | |d_c|^2] (one 19 KB collective; any rank-consistent choice within rounding would do).
      VGG_CUDA_CHECK(cudaMemcpyAsync(L.d_c + L.Dpad - 2, L.scal, sizeof(double) * 2, cudaMemcpyDeviceToDevice, st));
      if ((rc = allreduce(ar_user, L.d_c, (size_t)L.Dpad, 1, st))) return rc;
      VGG_CUDA_CHECK(cudaMemcpyAsync(L.scal, L.d_c + L.Dpad - 2, sizeof(double) * 2, cudaMemcpyDeviceToDevice, st));
    }
    if ((rc = launch_backsub(D, N, L.blk[cur].W, L.d_c, L.wacc, st))) return rc;
    if ((rc = launch_point_step(N, L.M, L.blk[cur].g_p, L.wacc, L.sc_p, L.dpp, L.points[cur], radius, L.points[cand],
                                L.scal, st)))
      return rc;
    if ((rc = launch_cam_update(S, dc, ns, prob->camera_model, L.d_c, L.poses[cur], L.intr[cur], L.poses[cand],
                                L.intr[cand], st)))
      return rc;
    if ((rc = eval(cand))) return rc;
    // point-side model terms join the candidate cost in the small all-reduce
    VGG_CUDA_CHECK(cudaMemsetAsync(L.small, 0, sizeof(double) * (8 + (size_t)L.Dpad), st));
    VGG_CUDA_CHECK(cudaMemcpyAsync(L.small, L.blk[cand].cost, sizeof(double), cudaMemcpyDeviceToDevice, st));
    VGG_CUDA_CHECK(cudaMemcpyAsync(L.small + 1, L.scal + 2, sizeof(double) * 2, cudaMemcpyDeviceToDevice, st));
    VGG_CUDA_CHECK(cudaMemcpyAsync(L.small + 3, L.scal + 6, sizeof(double), cudaMemcpyDeviceToDevice, st));
    if ((rc = launch_extract_gvec(S, dc, ns, L.KR, L.blk[cand].camrec, L.blk[cand].shared, L.small + 8, st))) return rc;
    if (fab2.on) {
      // one in-kernel all-reduce for everything: the point-gradient max rides in slot 4 (max), the rest is summed
      if ((rc = launch_gradmax(D, N, L.small + 8, prob->param_const, L.blk[cand].g_p, prob->point_const, L.scal, st))) return rc;
      VGG_CUDA_CHECK(cudaMemcpyAsync(L.small + 4, L.scal + 5, sizeof(double), cudaMemcpyDeviceToDevice, st));
      if ((rc = fab2.allreduce(L.small, 8 + L.Dpad, 4, st))) return rc;
      VGG_CUDA_CHECK(cudaMemsetAsync(L.scal + 4, 0, sizeof(double) * 2, st));
      if ((rc = launch_gradmax(D, N, L.small + 8, prob->param_const, L.blk[cand].g_p, prob->point_const, L.scal, st))) return rc;
      VGG_CUDA_CHECK(cudaMemcpyAsync(L.scal + 5, L.small + 4, sizeof(double), cudaMemcpyDeviceToDevice, st));
    } else {
      if (allreduce && (rc = allreduce(ar_user, L.small, 8 + (size_t)L.Dpad, 0, st))) return rc;
      if ((rc = launch_gradmax(D, N, L.small + 8, prob->param_const, L.blk[cand].g_p, prob->point_const, L.scal, st))) return rc;
      if (allreduce && (rc = allreduce(ar_user, L.scal + 5, 1, 1, st))) return rc;
    }
    if (opt.parameter_tolerance > 0.0) {
      // |x| of THIS rank's points + the replicated cameras; with track shards the point part is a partial sum, which
      // only makes the test stricter by under-estimating |x| (parameter_tolerance is 0 in every COLMAP preset)
      xnorm_kernel<<<1, 1024, 0, st>>>(S, N, dc, ns, prob->camera_model, prob->param_const, prob->point_const,
                                        L.poses[cur], L.intr[cur], L.points[cur], L.scal + 8);
      VGG_LAUNCH_CHECK();
    }
    if ((rc = read_scalars())) return rc;

    const double c_cost = h_scal[8];
    const double quad = h_scal[0] + h_scal[9];
    const double step_norm = sqrt(h_scal[1] + h_scal[10]);
    const double model_change = 0.5 * quad;
    if (h_scal[19] != 0.0) {
      set_error("fabric barrier timed out: a peer rank did not arrive");
      return VGG_ECUDA;
    }
    const bool solver_bad = h_scal[16] != 0.0 || h_scal[7] > 0 || h_scal[11] > 0;
    double* tr = trace ? trace + (size_t)(it - 1) * 8 : nullptr;
    if (tr) {
      tr[0] = it; tr[1] = cost; tr[2] = c_cost; tr[3] = model_change; tr[4] = 0; tr[5] = radius; tr[6] = step_norm; tr[7] = 0;
    }
    if (solver_bad || !(model_change > 0.0) || !isfinite(c_cost)) {
      // Ceres: invalid step -> LevenbergMarquardtStrategy::StepIsInvalid
      ++invalid_steps;
      if (tr) tr[7] = 2;
      if (invalid_steps >= opt.max_num_consecutive_invalid_steps) {
        summary->termination = VGG_BA_FAILURE;
        break;
      }
      radius *= 0.5;
      continue;
    }
    invalid_steps = 0;
    const double cost_change = cost - c_cost;
    const double rho = cost_change / model_change;
    if (tr) tr[4] = rho;
    // Ceres ParameterToleranceReached(): step_norm <= tol * (|x| + tol), |x| over the non-constant blocks in ambient
    // coordinates (h_scal[18], xnorm_kernel; only evaluated when the tolerance is non-zero -- COLMAP's default is 0)
    const double x_norm = opt.parameter_tolerance > 0.0 ? sqrt(h_scal[18]) : 0.0;
    if (step_norm <= opt.parameter_tolerance * (x_norm + opt.parameter_tolerance)) {
      summary->termination = VGG_BA_CONVERGENCE_PARAMETER;
      break;
    }
    const bool success = rho > opt.min_relative_decrease;
    if (fabs(cost_change) <= opt.function_tolerance * cost) {
      // Ceres 2.x TrustRegionMinimizer::Minimize returns from FunctionToleranceReached() before IsStepSuccessful() /
      // HandleSuccessfulStep(): the candidate of the terminating iteration is discarded
      summary->termination = VGG_BA_CONVERGENCE_FUNCTION;
      break;
    }
    if (success) {
      cur = cand;
      cost = c_cost;
      summary->successful++;
      if (tr) tr[7] = 1;
      radius = fmin(opt.max_trust_region_radius, radius / fmax(1.0 / 3.0, 1.0 - pow(2.0 * rho - 1.0, 3.0)));
      decrease_factor = 2.0;
      gmax = fmax(h_scal[4], h_scal[5]);
      if (gmax <= opt.gradient_tolerance) {
        summary->termination = VGG_BA_CONVERGENCE_GRADIENT;
        break;
      }
    } else {
      radius = radius / decrease_factor;
      decrease_factor *= 2.0;
    }
  }

  VGG_CUDA_CHECK(cudaMemcpyAsync(prob->poses, L.poses[cur], sizeof(double) * (size_t)S * 12, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemcpyAsync(prob->intr, L.intr[cur], sizeof(double) * (size_t)S * 4, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaMemcpyAsync(prob->points, L.points[cur], sizeof(double) * (size_t)N * 3, cudaMemcpyDeviceToDevice, st));
  VGG_CUDA_CHECK(cudaEventRecord(ev1, st));
  VGG_CUDA_CHECK(cudaEventSynchronize(ev1));
  float ms = 0;
  VGG_CUDA_CHECK(cudaEventElapsedTime(&ms, ev0, ev1));
  summary->iterations = it;
  summary->final_cost = cost;
  summary->final_radius = radius;
  summary->device_ms = ms;
  summary->kernel_launches = g_launch_count;
  return VGG_OK;
}

}  // extern "C"
