// HED soft-edge annotator of ControlNet.preprocess(type='hed' / 'softedge_v11p') on the GPU.
//
// Replaces controlnet.py:370-376 -> controlnet_annotator/hed/__init__.py:102-128 (ControlNetHED_Apache2 in fp32 on
// the raw 0-255 image, five projections copied to the host, cv2.resize + mean + sigmoid on the CPU per image).
// The 13 3x3 convs run on the tcgen05 implicit GEMM (pfd_gemm_f16, fp16 storage, fp32 accumulation); this file holds
// the pieces around them:
//   hed_input    ToPILImage quantisation, (u8 - norm[c]) * scale -> channel-last fp16.  norm is subtracted before the
//                stem's zero padding (the reference pads x - norm, so it cannot be folded into the first bias);
//                `scale` is the power-of-two activation scale the caller folded into every conv bias;
//   maxpool2x2   channel-last 2x2 / stride 2 max-pool with floor semantics (odd sizes drop the last row / column);
//   hed_project  the 1x1 conv to one channel, fp32 dot product per pixel (reads the activation once) -> fp32 logits;
//   hed_fuse     five logit maps -> INTER_LINEAR resize (cv2.resize) -> float32 mean -> float64 sigmoid -> x255, clip,
//                truncate -> ToTensor -> float32 [B,3,H,W]; counts non-finite mean logits (fp16 overflow guard).
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/pfd_b200.h"
#include "common.h"
#include "image_u8.cuh"

namespace pfd {

__device__ __forceinline__ void pdl_enter_h() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

static inline int grid_1d(long long total, int per_cta) {
  long long g = (total + per_cta - 1) / per_cta;
  const long long cap = (long long)num_sms() * 16;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

template <typename T>
__global__ void hed_input_kernel(const T* __restrict__ x, int B, int H, int W, const float* __restrict__ norm,
                                 float scale, __half* __restrict__ out) {
  pdl_enter_h();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  const float n0 = norm[0], n1 = norm[1], n2 = norm[2];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw, p = i % hw;
    const T* src = x + n * 3 * hw + p;
    __half* o = out + i * 3;
    o[0] = __float2half_rn(((float)to_u8<T>(src[0]) - n0) * scale);
    o[1] = __float2half_rn(((float)to_u8<T>(src[hw]) - n1) * scale);
    o[2] = __float2half_rn(((float)to_u8<T>(src[2 * hw]) - n2) * scale);
  }
}

__global__ void maxpool2x2_kernel(const uint4* __restrict__ x, int NB, int H, int W, int vecs, uint4* __restrict__ out) {
  pdl_enter_h();
  const int Ho = H / 2, Wo = W / 2;
  const long long total = (long long)NB * Ho * Wo * vecs;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % vecs);
    long long p = i / vecs;
    const int ox = (int)(p % Wo);
    p /= Wo;
    const int oy = (int)(p % Ho);
    const long long n = p / Ho;
    const uint4* r0 = x + ((n * H + 2 * oy) * W + 2 * ox) * vecs + v;
    const uint4* r1 = r0 + (long long)W * vecs;
    uint4 a = __ldg(r0), b = __ldg(r0 + vecs), c = __ldg(r1), d = __ldg(r1 + vecs);
    __half2* ha = reinterpret_cast<__half2*>(&a);
    const __half2* hb = reinterpret_cast<const __half2*>(&b);
    const __half2* hc = reinterpret_cast<const __half2*>(&c);
    const __half2* hd = reinterpret_cast<const __half2*>(&d);
#pragma unroll
    for (int k = 0; k < 4; ++k) ha[k] = __hmax2_nan(__hmax2_nan(ha[k], hb[k]), __hmax2_nan(hc[k], hd[k]));  // NaN propagates, as in F.max_pool2d
    out[i] = a;
  }
}

// G lanes (a power of two <= 32) share one pixel: lane j reads 16-byte channel vectors j, j+G, ... (coalesced), the
// partial dot products meet in a shuffle reduction.  out = dot(x, w) * inv_scale + b.
__global__ void __launch_bounds__(256)
hed_project_kernel(const uint4* __restrict__ x, long long M, int vecs, int G, const float4* __restrict__ w,
                   const float* __restrict__ b, float inv_scale, float* __restrict__ out) {
  pdl_enter_h();
  const int per_cta = blockDim.x / G;
  const int sub = threadIdx.x % G;
  const float bias = b[0];
  for (long long base = (long long)blockIdx.x * per_cta; base < M; base += (long long)gridDim.x * per_cta) {
    const long long m = base + threadIdx.x / G;
    float acc = 0.f;
    if (m < M) {
      const uint4* row = x + m * vecs;
      for (int v = sub; v < vecs; v += G) {
        const uint4 u = __ldg(row + v);
        const float4 w0 = __ldg(w + 2 * v), w1 = __ldg(w + 2 * v + 1);
        const __half2* h = reinterpret_cast<const __half2*>(&u);
        const float2 f0 = __half22float2(h[0]), f1 = __half22float2(h[1]);
        const float2 f2 = __half22float2(h[2]), f3 = __half22float2(h[3]);
        acc = fmaf(f0.x, w0.x, acc);
        acc = fmaf(f0.y, w0.y, acc);
        acc = fmaf(f1.x, w0.z, acc);
        acc = fmaf(f1.y, w0.w, acc);
        acc = fmaf(f2.x, w1.x, acc);
        acc = fmaf(f2.y, w1.y, acc);
        acc = fmaf(f3.x, w1.z, acc);
        acc = fmaf(f3.y, w1.w, acc);
      }
    }
    for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (m < M && sub == 0) out[m] = fmaf(acc, inv_scale, bias);
  }
}

struct FuseMaps {
  const float* p[PFD_HED_MAPS];
  int h[PFD_HED_MAPS], w[PFD_HED_MAPS];
  double sy[PFD_HED_MAPS], sx[PFD_HED_MAPS];   // source / destination size, as cv2 computes it (1 / inv_scale)
};

// INTER_LINEAR tap of cv2.resize on float32: half-pixel centre f = (d + 0.5) * scale - 0.5 in fp64, source index
// floor(f) and weights (1 - w, w) of w = f - floor(f) rounded to fp32; clamped to the first / last source index with
// weight 0 outside.
__device__ __forceinline__ void linear_tap(int d, double scale, int n, int& i0, int& i1, float& a0, float& a1) {
  const double f = (d + 0.5) * scale - 0.5;
  int i = (int)floor(f);
  double w = f - i;
  if (i < 0) {
    i = 0;
    w = 0.0;
  }
  if (i >= n - 1) {
    i = n - 1;
    w = 0.0;
  }
  i0 = i;
  i1 = min(i + 1, n - 1);
  a0 = (float)(1.0 - w);
  a1 = (float)w;
}

__global__ void hed_fuse_kernel(FuseMaps maps, int B, int H, int W, float* __restrict__ out, int* __restrict__ nonfinite) {
  pdl_enter_h();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw, p = i % hw;
    const int y = (int)(p / W), xw = (int)(p % W);
    float acc = 0.f;
#pragma unroll
    for (int k = 0; k < PFD_HED_MAPS; ++k) {
      int y0, y1, x0, x1;
      float b0, b1, a0, a1;
      linear_tap(y, maps.sy[k], maps.h[k], y0, y1, b0, b1);
      linear_tap(xw, maps.sx[k], maps.w[k], x0, x1, a0, a1);
      const float* src = maps.p[k] + n * maps.h[k] * maps.w[k];
      const float* r0 = src + (long long)y0 * maps.w[k];
      const float* r1 = src + (long long)y1 * maps.w[k];
      // unfused products, rows first, as cv2's separable float path
      const float h0 = __fadd_rn(__fmul_rn(__ldg(r0 + x0), a0), __fmul_rn(__ldg(r0 + x1), a1));
      const float h1 = __fadd_rn(__fmul_rn(__ldg(r1 + x0), a0), __fmul_rn(__ldg(r1 + x1), a1));
      acc = __fadd_rn(acc, __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1)));
    }
    const float mean = __fdiv_rn(acc, (float)PFD_HED_MAPS);      // np.mean of float32: float32 sum / count
    float v = 0.f;
    if (isfinite(mean)) {
      double e = 1.0 / (1.0 + exp(-(double)mean)) * 255.0;
      e = fmin(fmax(e, 0.0), 255.0);
      v = (float)(int)e / 255.f;                                     // astype(uint8) truncates; ToTensor divides
    } else {
      atomicAdd(nonfinite, 1);
    }
    float* o = out + n * 3 * hw + p;
    o[0] = v;
    o[hw] = v;
    o[2 * hw] = v;
  }
}

}  // namespace pfd

using namespace pfd;

extern "C" PFD_API int pfd_hed_input_f16(const void* x, int32_t src_is_f32, int32_t B, int32_t H, int32_t W,
                                         const float* norm, float scale, void* out, void* stream) {
  if (!x || !norm || !out || B <= 0 || H <= 0 || W <= 0) return set_error("pfd_hed_input_f16: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = (long long)B * H * W;
  if (src_is_f32)
    launch_k(hed_input_kernel<float>, dim3(grid_1d(total, 256)), dim3(256), (size_t)0, st, static_cast<const float*>(x),
             (int)B, (int)H, (int)W, norm, scale, static_cast<__half*>(out));
  else
    launch_k(hed_input_kernel<__half>, dim3(grid_1d(total, 256)), dim3(256), (size_t)0, st, static_cast<const __half*>(x),
             (int)B, (int)H, (int)W, norm, scale, static_cast<__half*>(out));
  return check_launch("hed_input");
}

extern "C" PFD_API int pfd_maxpool2x2_f16(const void* x, int32_t NB, int32_t H, int32_t W, int32_t C, void* out,
                                          void* stream) {
  if (!x || !out || NB <= 0 || H < 2 || W < 2 || C <= 0 || C % 8)
    return set_error("pfd_maxpool2x2_f16: bad arguments (NB=%d H=%d W=%d C=%d)", NB, H, W, C);
  const long long total = (long long)NB * (H / 2) * (W / 2) * (C / 8);
  launch_k(maxpool2x2_kernel, dim3(grid_1d(total, 256)), dim3(256), (size_t)0, static_cast<cudaStream_t>(stream),
           static_cast<const uint4*>(x), (int)NB, (int)H, (int)W, (int)(C / 8), static_cast<uint4*>(out));
  return check_launch("maxpool2x2");
}

extern "C" PFD_API int pfd_hed_project_f32(const void* x, int64_t M, int32_t C, const float* w, const float* b,
                                           float inv_scale, float* out, void* stream) {
  if (!x || !w || !b || !out || M <= 0 || C <= 0 || C % 8)
    return set_error("pfd_hed_project_f32: bad arguments (M=%lld C=%d)", (long long)M, C);
  const int vecs = C / 8;
  int G = 1;
  while (G * 2 <= vecs && G < 32) G *= 2;
  launch_k(hed_project_kernel, dim3(grid_1d(M, 256 / G)), dim3(256), (size_t)0, static_cast<cudaStream_t>(stream),
           static_cast<const uint4*>(x), (long long)M, vecs, G, reinterpret_cast<const float4*>(w), b, inv_scale, out);
  return check_launch("hed_project");
}

extern "C" PFD_API int pfd_hed_fuse_f32(const float* const* maps, const int32_t* map_h, const int32_t* map_w,
                                        int32_t B, int32_t H, int32_t W, float* out, int32_t* nonfinite,
                                        void* stream) {
  if (!maps || !map_h || !map_w || !out || !nonfinite || B <= 0 || H <= 0 || W <= 0)
    return set_error("pfd_hed_fuse_f32: bad arguments");
  FuseMaps fm;
  for (int k = 0; k < PFD_HED_MAPS; ++k) {
    if (!maps[k] || map_h[k] <= 0 || map_w[k] <= 0 || map_h[k] > H || map_w[k] > W)
      return set_error("pfd_hed_fuse_f32: map %d is %dx%d for a %dx%d output", k, map_h[k], map_w[k], H, W);
    fm.p[k] = maps[k];
    fm.h[k] = map_h[k];
    fm.w[k] = map_w[k];
    fm.sy[k] = 1.0 / ((double)H / map_h[k]);
    fm.sx[k] = 1.0 / ((double)W / map_w[k]);
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(nonfinite, 0, sizeof(int32_t), st) != cudaSuccess)
    return set_error("pfd_hed_fuse_f32: memset failed: %s", cudaGetErrorString(cudaGetLastError()));
  launch_k(hed_fuse_kernel, dim3(grid_1d((long long)B * H * W, 256)), dim3(256), (size_t)0, st, fm, (int)B, (int)H,
           (int)W, out, reinterpret_cast<int*>(nonfinite));
  return check_launch("hed_fuse");
}
