// Fused correlation + local sampling for the track predictor's inner loop.
//
// Replaces CorrBlock.corr + CorrBlock.sample (vggsfm/models/track_modules/blocks.py:363-416, called every
// refinement iteration from base_track_predictor.py:135-139) and EfficientCorrBlock.sample (:433-471).
// The reference multiplies every target feature with EVERY spatial position of every pyramid level
// ([B,S,N,C] x [B,S,C,H*W], 21 824 positions per (frame, query) in the coarse tracker), writes the volume
// to HBM and then bilinearly samples (2r+1)^2 taps per level from it.  All taps of one (frame, query, level)
// share one fractional offset, so the sampled values only depend on the (2r+2)^2 integer positions around
// the query: this kernel computes exactly those dot products (44x fewer MACs for r=4 on a 128^2 map) from a
// channels-last pyramid (one coalesced C-vector per position) and interpolates in registers.  The
// correlation volume never exists.  grid_sample semantics kept: align_corners=True, padding "zeros"
// (CorrBlock) or "border" (EfficientCorrBlock), tap order out[a*(2r+1)+b] with x = cx + (a-r), y = cy + (b-r)
// (blocks.py:374-382).
#include <cuda_fp16.h>
#include "common.cuh"

namespace vgg {

// ---- pyramid construction: NCHW float -> NHWC (float, optionally also half), then 2x2 average pooling ----
template <typename TOUT>
__global__ void nchw_to_nhwc_kernel(int C, int H, int W, const float* __restrict__ in, float* __restrict__ out32,
                                    TOUT* __restrict__ outT) {
  // grid: (ceil(HW/32) * images, ceil(C/32)); block (32, 8)   (images in x: the fine tracker has 131 072 of them)
  __shared__ float tile[32][33];
  const int HW = H * W;
  const int tiles_hw = (HW + 31) / 32;
  const size_t img = blockIdx.x / tiles_hw;
  const int p0 = (int)(blockIdx.x % tiles_hw) * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int c = c0 + j, p = p0 + threadIdx.x;
    tile[j][threadIdx.x] = (c < C && p < HW) ? in[(img * C + c) * HW + p] : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int p = p0 + j, c = c0 + threadIdx.x;
    if (p < HW && c < C) {
      const float v = tile[threadIdx.x][j];
      if (out32) out32[(img * HW + p) * C + c] = v;
      if (outT) outT[(img * HW + p) * C + c] = (TOUT)v;
    }
  }
}

template <typename TOUT>
__global__ void pool_nhwc_kernel(int C, int H, int W, const float* __restrict__ in, float* __restrict__ out32,
                                 TOUT* __restrict__ outT, size_t total) {
  const int Ho = H / 2, Wo = W / 2;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  size_t r = i / C;
  const int x = (int)(r % Wo); r /= Wo;
  const int y = (int)(r % Ho);
  const size_t img = r / Ho;
  const float* base = in + ((img * H + 2 * y) * W + 2 * x) * C + c;
  const float v = (base[0] + base[C] + base[(size_t)W * C] + base[(size_t)W * C + C]) * 0.25f;
  if (out32) out32[i] = v;
  if (outT) outT[i] = (TOUT)v;
}

struct CorrLevels {
  const void* fmap[8];   // NHWC level pointers
  int H[8], W[8];
};

template <typename T> struct VecLoad;
template <> struct VecLoad<float> {
  template <int CPL>
  static __device__ __forceinline__ void load(const float* p, float* o) {
    if constexpr (CPL == 4) { const float4 v = *reinterpret_cast<const float4*>(p); o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
    else if constexpr (CPL == 2) { const float2 v = *reinterpret_cast<const float2*>(p); o[0] = v.x; o[1] = v.y; }
    else { for (int i = 0; i < CPL; ++i) o[i] = p[i]; }
  }
};
template <> struct VecLoad<__half> {
  template <int CPL>
  static __device__ __forceinline__ void load(const __half* p, float* o) {
    if constexpr (CPL == 4) {
      const uint2 v = *reinterpret_cast<const uint2*>(p);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
      o[0] = a.x; o[1] = a.y; o[2] = b.x; o[3] = b.y;
    } else if constexpr (CPL == 2) {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(p));
      o[0] = a.x; o[1] = a.y;
    } else { for (int i = 0; i < CPL; ++i) o[i] = __half2float(p[i]); }
  }
};

// one warp per (image = b*S+s, query n); lanes over channels (CPL channels per lane, C = 32*CPL)
template <typename T, int CPL, int R>
__global__ void __launch_bounds__(256) corr_sample_kernel(int BS, int N, int L, CorrLevels lv,
                                                          const float* __restrict__ targets /*[BS,N,C]*/,
                                                          const float* __restrict__ coords /*[BS,N,2]*/, int border,
                                                          float* __restrict__ out /*[BS,N,L*(2R+1)^2]*/) {
  constexpr int C = 32 * CPL;
  constexpr int FP = 2 * R + 2;          // footprint side
  constexpr int NF = FP * FP;            // footprint positions
  constexpr int NG = (NF + 31) / 32;     // reduce groups
  constexpr int K = 2 * R + 1;
  __shared__ float dsm[8][NG * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t q = (size_t)blockIdx.x * 8 + warp;
  if (q >= (size_t)BS * N) return;
  const size_t img = q / N;
  float tg[CPL];
  {
    const float* tp = targets + q * C + lane * CPL;
#pragma unroll
    for (int i = 0; i < CPL; ++i) tg[i] = (float)(T)tp[i];       // round to the pyramid precision like autocast does
  }
  const float cx0 = coords[q * 2], cy0 = coords[q * 2 + 1];
  const float inv_sqrt_c = rsqrtf((float)C);
  float* orow = out + q * (size_t)L * K * K;
  for (int l = 0; l < L; ++l) {
    const int H = lv.H[l], W = lv.W[l];
    const T* fm = reinterpret_cast<const T*>(lv.fmap[l]) + img * (size_t)H * W * C;
    const float scale = 1.0f / (float)(1 << l);
    // reference: coords/2^l + delta, then x*(2/(W-1)) - 1 and grid_sample's un-normalisation ((x+1)/2*(W-1))
    const float cx = cx0 * scale, cy = cy0 * scale;
    const float fxf = floorf(cx), fyf = floorf(cy);
    const int fx = (int)fxf, fy = (int)fyf;
    // Every footprint position is loaded UNCONDITIONALLY from a clamped address and masked afterwards: the loads of a
    // level are then independent straight-line code the compiler issues back to back.  (r02 measurement of the guarded
    // version, one `if (inside) load` per position: the 64-192 loads of a query serialised on their latency -- 4.2 ms
    // for the fine tracker's 131 072 patches, 6 % of the HBM roofline.)
    float part[NF];
#pragma unroll
    for (int iy = 0; iy < FP; ++iy) {
      const int Y = fy - R + iy;
      const bool yin = border || (Y >= 0 && Y < H);
      const int Yc = min(max(Y, 0), H - 1);
#pragma unroll
      for (int ix = 0; ix < FP; ++ix) {
        const int X = fx - R + ix;
        const bool xin = border || (X >= 0 && X < W);
        const int Xc = min(max(X, 0), W - 1);
        float f[CPL];
        VecLoad<T>::template load<CPL>(fm + ((size_t)Yc * W + Xc) * C + lane * CPL, f);
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < CPL; ++i) acc = fmaf(tg[i], f[i], acc);
        part[iy * FP + ix] = (yin && xin) ? acc : 0.f;
      }
    }
    // warp reduce-scatter in groups of 32 footprint positions
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      float v[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = (g * 32 + i < NF) ? part[(g * 32 + i < NF) ? g * 32 + i : 0] : 0.f;
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
          const float mine = up ? v[i + off] : v[i];
          const float send = up ? v[i] : v[i + off];
          v[i] = mine + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      dsm[warp][g * 32 + lane] = v[0] * inv_sqrt_c;
    }
    __syncwarp();
    // bilinear interpolation of the K*K taps
    for (int o = lane; o < K * K; o += 32) {
      const int a = o / K, b = o % K;
      float x = cx + (float)(a - R), y = cy + (float)(b - R);
      float val;
      if (!border) {
        const float wx = cx - fxf, wy = cy - fyf;        // same fraction for every tap
        const int ix = a, iy = b;                        // footprint index of floor(x), floor(y)
        const float d00 = dsm[warp][iy * FP + ix], d01 = dsm[warp][iy * FP + ix + 1];
        const float d10 = dsm[warp][(iy + 1) * FP + ix], d11 = dsm[warp][(iy + 1) * FP + ix + 1];
        val = d00 * (1.f - wx) * (1.f - wy) + d01 * wx * (1.f - wy) + d10 * (1.f - wx) * wy + d11 * wx * wy;
      } else {
        x = fminf(fmaxf(x, 0.f), (float)(W - 1));
        y = fminf(fmaxf(y, 0.f), (float)(H - 1));
        const float x0f = floorf(x), y0f = floorf(y);
        const float wx = x - x0f, wy = y - y0f;
        const int x0 = (int)x0f, y0 = (int)y0f;
        const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
        // footprint slot i holds position clamp(f - R + i): invert (monotone) by clamping the slot index
        auto slotx = [&](int X) { return min(max(X - (fx - R), 0), FP - 1); };
        auto sloty = [&](int Y) { return min(max(Y - (fy - R), 0), FP - 1); };
        const float d00 = dsm[warp][sloty(y0) * FP + slotx(x0)], d01 = dsm[warp][sloty(y0) * FP + slotx(x1)];
        const float d10 = dsm[warp][sloty(y1) * FP + slotx(x0)], d11 = dsm[warp][sloty(y1) * FP + slotx(x1)];
        val = d00 * (1.f - wx) * (1.f - wy) + d01 * wx * (1.f - wy) + d10 * (1.f - wx) * wy + d11 * wx * wy;
      }
      orow[(size_t)l * K * K + o] = val;
    }
    __syncwarp();
  }
}

// C = 32 (the fine tracker's patch pyramids): lanes over FOOTPRINT POSITIONS instead of channels.  With one channel per
// lane every position was one 64-byte load per warp instruction (half pyramid) followed by a 32-lane reduce-scatter --
// r02 ncu: 146 registers, one CTA per SM, issue slots 46 %, 2 TB/s.  Here a lane owns positions lane, lane + 32, ...:
// it loads the position's whole 32-channel vector with 16-byte loads (8 neighbouring positions = 512 contiguous bytes),
// keeps the 32 target values in registers and writes the finished dot product -- no shuffles at all.
template <typename T> struct Vec32;
template <> struct Vec32<float> {
  static __device__ __forceinline__ float dot(const float* __restrict__ p, const float (&tg)[32]) {
    float acc = 0.f;
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const float4 f = *reinterpret_cast<const float4*>(p + 4 * v);
      acc = fmaf(tg[4 * v], f.x, acc);
      acc = fmaf(tg[4 * v + 1], f.y, acc);
      acc = fmaf(tg[4 * v + 2], f.z, acc);
      acc = fmaf(tg[4 * v + 3], f.w, acc);
    }
    return acc;
  }
};
template <> struct Vec32<__half> {
  static __device__ __forceinline__ float dot(const __half* __restrict__ p, const float (&tg)[32]) {
    float acc = 0.f;
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      const uint4 raw = *reinterpret_cast<const uint4*>(p + 8 * v);
      const __half2* h = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __half22float2(h[i]);
        acc = fmaf(tg[8 * v + 2 * i], f.x, acc);         // same summation order as the channel-per-lane kernel is NOT
        acc = fmaf(tg[8 * v + 2 * i + 1], f.y, acc);     // kept (that one reduces across lanes); both are fp32 sums
      }
    }
    return acc;
  }
};

template <typename T, int R>
__global__ void __launch_bounds__(256, 4) corr_sample_c32_kernel(int BS, int N, int L, CorrLevels lv,
                                                                 const float* __restrict__ targets /*[BS,N,32]*/,
                                                                 const float* __restrict__ coords /*[BS,N,2]*/, int border,
                                                                 float* __restrict__ out /*[BS,N,L*(2R+1)^2]*/) {
  constexpr int C = 32;
  constexpr int FP = 2 * R + 2;          // footprint side
  constexpr int NF = FP * FP;            // footprint positions
  constexpr int NPL = (NF + 31) / 32;    // positions per lane
  constexpr int K = 2 * R + 1;
  __shared__ float dsm[8][NPL * 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t q = (size_t)blockIdx.x * 8 + warp;
  if (q >= (size_t)BS * N) return;
  const size_t img = q / N;
  float tg[C];
  {
    const float4* tp = reinterpret_cast<const float4*>(targets + q * C);
#pragma unroll
    for (int v = 0; v < 8; ++v) {
      const float4 t = tp[v];
      tg[4 * v] = (float)(T)t.x;          // round to the pyramid precision like autocast does
      tg[4 * v + 1] = (float)(T)t.y;
      tg[4 * v + 2] = (float)(T)t.z;
      tg[4 * v + 3] = (float)(T)t.w;
    }
  }
  const float cx0 = coords[q * 2], cy0 = coords[q * 2 + 1];
  const float inv_sqrt_c = rsqrtf((float)C);
  float* orow = out + q * (size_t)L * K * K;
  for (int l = 0; l < L; ++l) {
    const int H = lv.H[l], W = lv.W[l];
    const T* fm = reinterpret_cast<const T*>(lv.fmap[l]) + img * (size_t)H * W * C;
    const float scale = 1.0f / (float)(1 << l);
    const float cx = cx0 * scale, cy = cy0 * scale;
    const float fxf = floorf(cx), fyf = floorf(cy);
    const int fx = (int)fxf, fy = (int)fyf;
#pragma unroll
    for (int s = 0; s < NPL; ++s) {
      const int p = s * 32 + lane;
      const int iy = p / FP, ix = p - iy * FP;
      const int Y = fy - R + iy, X = fx - R + ix;
      const bool in = p < NF && (border || (Y >= 0 && Y < H && X >= 0 && X < W));
      const int Yc = min(max(Y, 0), H - 1), Xc = min(max(X, 0), W - 1);     // unconditional load from a clamped address
      const float acc = Vec32<T>::dot(fm + ((size_t)Yc * W + Xc) * C, tg);
      dsm[warp][p] = in ? acc * inv_sqrt_c : 0.f;
    }
    __syncwarp();
    // bilinear interpolation of the K*K taps (identical to corr_sample_kernel)
    for (int o = lane; o < K * K; o += 32) {
      const int a = o / K, b = o % K;
      float x = cx + (float)(a - R), y = cy + (float)(b - R);
      float val;
      if (!border) {
        const float wx = cx - fxf, wy = cy - fyf;
        const int ix = a, iy = b;
        const float d00 = dsm[warp][iy * FP + ix], d01 = dsm[warp][iy * FP + ix + 1];
        const float d10 = dsm[warp][(iy + 1) * FP + ix], d11 = dsm[warp][(iy + 1) * FP + ix + 1];
        val = d00 * (1.f - wx) * (1.f - wy) + d01 * wx * (1.f - wy) + d10 * (1.f - wx) * wy + d11 * wx * wy;
      } else {
        x = fminf(fmaxf(x, 0.f), (float)(W - 1));
        y = fminf(fmaxf(y, 0.f), (float)(H - 1));
        const float x0f = floorf(x), y0f = floorf(y);
        const float wx = x - x0f, wy = y - y0f;
        const int x0 = (int)x0f, y0 = (int)y0f;
        const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
        auto slotx = [&](int X) { return min(max(X - (fx - R), 0), FP - 1); };
        auto sloty = [&](int Y) { return min(max(Y - (fy - R), 0), FP - 1); };
        const float d00 = dsm[warp][sloty(y0) * FP + slotx(x0)], d01 = dsm[warp][sloty(y0) * FP + slotx(x1)];
        const float d10 = dsm[warp][sloty(y1) * FP + slotx(x0)], d11 = dsm[warp][sloty(y1) * FP + slotx(x1)];
        val = d00 * (1.f - wx) * (1.f - wy) + d01 * wx * (1.f - wy) + d10 * (1.f - wx) * wy + d11 * wx * wy;
      }
      orow[(size_t)l * K * K + o] = val;
    }
    __syncwarp();
  }
}

template <typename T>
static int launch_corr(int BS, int N, int C, int L, int R, const CorrLevels& lv, const float* targets,
                       const float* coords, int border, float* out, cudaStream_t st) {
  const size_t nq = (size_t)BS * N;
  const unsigned grid = (unsigned)((nq + 7) / 8);
#define VGG_CORR_CASE(CPLV, RV)                                                                                    \
  if (C == 32 * CPLV && R == RV) {                                                                                 \
    corr_sample_kernel<T, CPLV, RV><<<grid, 256, 0, st>>>(BS, N, L, lv, targets, coords, border, out);             \
    VGG_LAUNCH_CHECK();                                                                                            \
    return VGG_OK;                                                                                                 \
  }
  // C = 32: position-per-lane kernel (0.35 ms against 1.01 ms for the channel-per-lane one on a B200,
  // DESIGN.md section 4.6); pointers must be 16-byte aligned, which every level of an NHWC pyramid with C = 32 is
  if (C == 32 && (R == 3 || R == 4) && (reinterpret_cast<uintptr_t>(targets) & 15) == 0) {
    bool aligned = true;
    for (int l = 0; l < L; ++l) aligned = aligned && (reinterpret_cast<uintptr_t>(lv.fmap[l]) & 15) == 0;
    if (aligned) {
      if (R == 3) corr_sample_c32_kernel<T, 3><<<grid, 256, 0, st>>>(BS, N, L, lv, targets, coords, border, out);
      else corr_sample_c32_kernel<T, 4><<<grid, 256, 0, st>>>(BS, N, L, lv, targets, coords, border, out);
      VGG_LAUNCH_CHECK();
      return VGG_OK;
    }
  }
  VGG_CORR_CASE(4, 4)   // coarse tracker: C=128, r=4
  VGG_CORR_CASE(4, 3)
  VGG_CORR_CASE(1, 3)   // fine tracker: C=32, r=3
  VGG_CORR_CASE(1, 4)
  VGG_CORR_CASE(2, 3)
  VGG_CORR_CASE(2, 4)
#undef VGG_CORR_CASE
  set_error("corr_sample: unsupported (C=%d, radius=%d); built for C in {32,64,128}, radius in {3,4}", C, R);
  return VGG_EINVAL;
}


// sample_features4d (vggsfm/models/utils.py:415-447): bilinear point sampling of an NCHW map with
// align_corners=True and border padding.  One warp per point, lanes stride the channels; the four taps of a
// channel are 4-byte gathers from one plane (NCHW is what the reference hands over; C is 3 for the colour
// read-back at models/triangulator.py:324 and 128 for the tracker's query features).
__global__ void sample_features_kernel(int B, int C, int H, int W, int R, const float* __restrict__ in,
                                       const float* __restrict__ coords, float* __restrict__ out) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (gw >= B * R) return;
  const int b = gw / R;
  float x = coords[(size_t)gw * 2], y = coords[(size_t)gw * 2 + 1];
  // grid_sample's unnormalise(normalise(x)) round trip, then the border clamp
  const float sx = 2.0f / (float)max(W - 1, 1), sy = 2.0f / (float)max(H - 1, 1);
  x = ((x * sx - 1.0f) + 1.0f) * 0.5f * (float)(W - 1);
  y = ((y * sy - 1.0f) + 1.0f) * 0.5f * (float)(H - 1);
  x = fminf(fmaxf(x, 0.0f), (float)(W - 1));
  y = fminf(fmaxf(y, 0.0f), (float)(H - 1));
  const float fx = floorf(x), fy = floorf(y);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, W - 1), y1 = min(y0 + 1, H - 1);
  const float ax = x - fx, ay = y - fy;
  const float w00 = (1.0f - ax) * (1.0f - ay), w01 = ax * (1.0f - ay), w10 = (1.0f - ax) * ay, w11 = ax * ay;
  const float* base = in + (size_t)b * C * H * W;
  for (int c = lane; c < C; c += 32) {
    const float* pl = base + (size_t)c * H * W;
    const float v = pl[(size_t)y0 * W + x0] * w00 + pl[(size_t)y0 * W + x1] * w01 + pl[(size_t)y1 * W + x0] * w10 +
                    pl[(size_t)y1 * W + x1] * w11;
    out[(size_t)gw * C + c] = v;
  }
}

}  // namespace vgg

using namespace vgg;

extern "C" {

// bytes of the channels-last pyramid (all levels) in the given element size, plus the float scratch
int vgg_corr_pyramid_bytes(int BS, int C, int H, int W, int num_levels, int elem_size, size_t* pyramid_bytes,
                           size_t* scratch_bytes) {
  VGG_REQUIRE(BS > 0 && C > 0 && H > 0 && W > 0 && num_levels >= 1 && num_levels <= 8, "bad sizes");
  VGG_REQUIRE(elem_size == 2 || elem_size == 4, "elem_size must be 2 (half) or 4 (float)");
  size_t tot = 0, tot32 = 0;
  int h = H, w = W;
  for (int l = 0; l < num_levels; ++l) {
    const size_t n = (size_t)BS * h * w * C;
    tot += align_up(n * elem_size, 256);
    tot32 += align_up(n * 4, 256);
    h /= 2; w /= 2;
    if (l + 1 < num_levels) VGG_REQUIRE(h > 0 && w > 0, "too many pyramid levels for this map size");
  }
  if (pyramid_bytes) *pyramid_bytes = tot;
  if (scratch_bytes) *scratch_bytes = (elem_size == 4) ? 0 : tot32;
  return VGG_OK;
}

int vgg_corr_build_pyramid(int BS, int C, int H, int W, int num_levels, const float* fmaps_nchw, int elem_size,
                           void* pyramid, void* scratch, void* stream) {
  VGG_REQUIRE(fmaps_nchw && pyramid, "null pointer");
  VGG_REQUIRE(elem_size == 4 || scratch, "half pyramid needs the float scratch");
  cudaStream_t st = (cudaStream_t)stream;
  g_launch_count = 0;
  char* pT = reinterpret_cast<char*>(pyramid);
  char* p32 = reinterpret_cast<char*>(scratch);
  int h = H, w = W, hp = H, wp = W;
  const float* prev32 = nullptr;
  for (int l = 0; l < num_levels; ++l) {
    const size_t n = (size_t)BS * h * w * C;
    float* cur32 = (elem_size == 4) ? reinterpret_cast<float*>(pT) : reinterpret_cast<float*>(p32);
    if (l == 0) {
      dim3 grid((unsigned)((size_t)((h * w + 31) / 32) * BS), (C + 31) / 32), block(32, 8);
      if (elem_size == 4) nchw_to_nhwc_kernel<float><<<grid, block, 0, st>>>(C, h, w, fmaps_nchw, cur32, nullptr);
      else nchw_to_nhwc_kernel<__half><<<grid, block, 0, st>>>(C, h, w, fmaps_nchw, cur32, reinterpret_cast<__half*>(pT));
    } else {
      const unsigned grid = (unsigned)((n + 255) / 256);
      if (elem_size == 4) pool_nhwc_kernel<float><<<grid, 256, 0, st>>>(C, hp, wp, prev32, cur32, nullptr, n);
      else pool_nhwc_kernel<__half><<<grid, 256, 0, st>>>(C, hp, wp, prev32, cur32, reinterpret_cast<__half*>(pT), n);
    }
    VGG_LAUNCH_CHECK();
    prev32 = cur32;
    pT += align_up(n * elem_size, 256);
    if (elem_size != 4) p32 += align_up(n * 4, 256);
    hp = h; wp = w;
    h /= 2; w /= 2;
  }
  return VGG_OK;
}

int vgg_corr_sample(int BS, int N, int C, int H, int W, int num_levels, int radius, const void* pyramid, int elem_size,
                    const float* targets, const float* coords, int border_padding, float* out, void* stream) {
  VGG_REQUIRE(pyramid && targets && coords && out, "null pointer");
  VGG_REQUIRE(num_levels >= 1 && num_levels <= 8, "num_levels must be in [1,8]");
  cudaStream_t st = (cudaStream_t)stream;
  g_launch_count = 0;
  CorrLevels lv;
  const char* p = reinterpret_cast<const char*>(pyramid);
  int h = H, w = W;
  for (int l = 0; l < num_levels; ++l) {
    lv.fmap[l] = p;
    lv.H[l] = h; lv.W[l] = w;
    p += align_up((size_t)BS * h * w * C * elem_size, 256);
    h /= 2; w /= 2;
  }
  if (elem_size == 4) return launch_corr<float>(BS, N, C, num_levels, radius, lv, targets, coords, border_padding, out, st);
  return launch_corr<__half>(BS, N, C, num_levels, radius, lv, targets, coords, border_padding, out, st);
}

int vgg_sample_features4d(int B, int C, int H, int W, int R, const float* input_nchw, const float* coords, float* out,
                          void* stream) {
  VGG_REQUIRE(B >= 0 && C > 0 && H > 0 && W > 0 && R >= 0, "bad shape");
  g_launch_count = 0;
  if (B * R == 0) return VGG_OK;
  VGG_REQUIRE(input_nchw && coords && out, "null pointer");
  const long long warps = (long long)B * R;
  sample_features_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(B, C, H, W, R, input_nchw,
                                                                                              coords, out);
  VGG_LAUNCH_CHECK();
  return VGG_OK;
}

}  // extern "C"
