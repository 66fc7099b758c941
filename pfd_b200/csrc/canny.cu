// Canny edge pre-processing of the ControlNet control image on the GPU (SURVEY.md §8 f1).
//
// Replaces ControlNet.preprocess(type='canny') of the reference (controlnet.py:332-360): tensor -> ToPILImage
// (x.mul(255).byte()) -> cv2.Canny(img_rgb_u8, low, high) [controlnet_annotator/canny/__init__.py:4-5] ->
// ToTensor (/255) -> repeat to 3 channels -> float32.  cv2.Canny (OpenCV 4.x imgproc/canny.cpp, aperture 3,
// L2gradient = false) is pure integer work and is reproduced bit-exactly:
//   1. Sobel 3x3 dx, dy per colour channel with BORDER_REPLICATE (16-bit), magnitude |dx|+|dy|; per pixel the
//      channel with the largest magnitude wins (first one on ties);
//   2. non-maximum suppression with the fixed-point tan(22.5) / tan(67.5) sector test (TG22 = 13573, shift 15);
//      candidates (magnitude > low) are marked 0 (weak) or 2 (strong: magnitude > high), everything else 1;
//   3. hysteresis: weak pixels 8-connected to a strong pixel become strong (iterated tile-wise to the fixed
//      point, which is what the reference's stack-based flood fill computes);
//   4. edge = strong -> 1.0, written to all three output channels.
// These are HBM-bound byte kernels (a 512x512 image is 1 MB): one pixel per thread, 32-bit packed RGBX loads.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pfd_b200.h"
#include "common.h"
#include "image_u8.cuh"

namespace pfd {

__device__ __forceinline__ void pdl_enter_c() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

template <typename T>
__global__ void canny_pack_kernel(const T* __restrict__ x, int B, int H, int W, uint32_t* __restrict__ rgbx) {
  pdl_enter_c();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw, p = i % hw;
    const T* src = x + n * 3 * hw + p;
    rgbx[i] = to_u8<T>(src[0]) | (to_u8<T>(src[hw]) << 8) | (to_u8<T>(src[2 * hw]) << 16);
  }
}

// ToTensor(ToPILImage(x)): floor(x * 255) / 255 as float32 (controlnet.py:345-348, type 'input')
template <typename T>
__global__ void u8_roundtrip_kernel(const T* __restrict__ x, long long n, float* __restrict__ out) {
  pdl_enter_c();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (float)to_u8<T>(x[i]) / 255.f;
}

__global__ void canny_grad_kernel(const uint32_t* __restrict__ rgbx, int B, int H, int W,
                                  short2* __restrict__ dxy, unsigned short* __restrict__ mag) {
  pdl_enter_c();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw;
    const int y = (int)((i % hw) / W), xw = (int)(i % W);
    const uint32_t* img = rgbx + n * hw;
    const int ym = max(y - 1, 0), yp = min(y + 1, H - 1);          // BORDER_REPLICATE
    const int xm = max(xw - 1, 0), xp = min(xw + 1, W - 1);
    const uint32_t p00 = img[(long long)ym * W + xm], p01 = img[(long long)ym * W + xw], p02 = img[(long long)ym * W + xp];
    const uint32_t p10 = img[(long long)y * W + xm], p12 = img[(long long)y * W + xp];
    const uint32_t p20 = img[(long long)yp * W + xm], p21 = img[(long long)yp * W + xw], p22 = img[(long long)yp * W + xp];
    int bdx = 0, bdy = 0, bm = -1;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int sh = 8 * c;
      const int a00 = (p00 >> sh) & 255, a01 = (p01 >> sh) & 255, a02 = (p02 >> sh) & 255;
      const int a10 = (p10 >> sh) & 255, a12 = (p12 >> sh) & 255;
      const int a20 = (p20 >> sh) & 255, a21 = (p21 >> sh) & 255, a22 = (p22 >> sh) & 255;
      const int dx = (a02 - a00) + 2 * (a12 - a10) + (a22 - a20);
      const int dy = (a20 - a00) + 2 * (a21 - a01) + (a22 - a02);
      const int m = abs(dx) + abs(dy);
      if (m > bm) {                                                // strictly greater: first channel wins ties
        bm = m;
        bdx = dx;
        bdy = dy;
      }
    }
    dxy[i] = make_short2((short)bdx, (short)bdy);
    mag[i] = (unsigned short)bm;
  }
}

__global__ void canny_nms_kernel(const short2* __restrict__ dxy, const unsigned short* __restrict__ mag, int B, int H,
                                 int W, int low, int high, unsigned char* __restrict__ map) {
  pdl_enter_c();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw;
    const int y = (int)((i % hw) / W), xw = (int)(i % W);
    const unsigned short* mg = mag + n * hw;
    auto M = [&](int yy, int xx) -> int {                           // magnitude is zero outside the image
      return (yy < 0 || yy >= H || xx < 0 || xx >= W) ? 0 : (int)mg[(long long)yy * W + xx];
    };
    const int m = (int)mg[(long long)y * W + xw];
    unsigned char r = 1;
    if (m > low) {
      const short2 d = dxy[i];
      const int xs = d.x, ys = d.y;
      const int ax = abs(xs);
      const int ay = abs(ys) << 15;
      const int tg22x = ax * 13573;
      bool cand;
      if (ay < tg22x) {
        cand = (m > M(y, xw - 1)) && (m >= M(y, xw + 1));
      } else {
        const int tg67x = tg22x + (ax << 16);
        if (ay > tg67x) {
          cand = (m > M(y - 1, xw)) && (m >= M(y + 1, xw));
        } else {
          const int s = ((xs ^ ys) < 0) ? -1 : 1;
          cand = (m > M(y - 1, xw - s)) && (m > M(y + 1, xw + s));
        }
      }
      if (cand) r = (m > high) ? 2 : 0;
    }
    map[i] = r;
  }
}

// One hysteresis sweep: every 32x32 tile (with a 1-pixel halo) is iterated to its local fixed point in shared
// memory; *changed is raised when any pixel flipped so the host launches another sweep.
constexpr int HT = 32;
__global__ void __launch_bounds__(HT* HT)
canny_hyst_kernel(unsigned char* __restrict__ map, int H, int W, int* __restrict__ changed) {
  pdl_enter_c();
  __shared__ unsigned char t[HT + 2][HT + 2];
  unsigned char* img = map + (long long)blockIdx.z * H * W;
  const int x0 = blockIdx.x * HT, y0 = blockIdx.y * HT;
  const int tid = threadIdx.y * HT + threadIdx.x;
  for (int k = tid; k < (HT + 2) * (HT + 2); k += HT * HT) {
    const int ly = k / (HT + 2), lx = k % (HT + 2);
    const int gy = y0 + ly - 1, gx = x0 + lx - 1;
    t[ly][lx] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? img[(long long)gy * W + gx] : 1;
  }
  __syncthreads();
  const int ly = threadIdx.y + 1, lx = threadIdx.x + 1;
  bool mine = false;
  for (;;) {
    bool flip = false;
    if (t[ly][lx] == 0) {
      flip = t[ly - 1][lx - 1] == 2 || t[ly - 1][lx] == 2 || t[ly - 1][lx + 1] == 2 || t[ly][lx - 1] == 2 ||
             t[ly][lx + 1] == 2 || t[ly + 1][lx - 1] == 2 || t[ly + 1][lx] == 2 || t[ly + 1][lx + 1] == 2;
    }
    __syncthreads();
    if (flip) {
      t[ly][lx] = 2;
      mine = true;
    }
    if (!__syncthreads_or(flip)) break;
  }
  const int gy = y0 + threadIdx.y, gx = x0 + threadIdx.x;
  if (mine && gy < H && gx < W) {
    img[(long long)gy * W + gx] = 2;
    atomicExch(changed, 1);
  }
}

__global__ void canny_emit_kernel(const unsigned char* __restrict__ map, int B, int H, int W, float* __restrict__ out) {
  pdl_enter_c();
  const long long hw = (long long)H * W;
  const long long total = (long long)B * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / hw, p = i % hw;
    const float v = map[i] == 2 ? 1.f : 0.f;                         // 255 / 255 (ToTensor), repeated to RGB
    float* o = out + n * 3 * hw + p;
    o[0] = v;
    o[hw] = v;
    o[2 * hw] = v;
  }
}

static inline int grid1d(long long total) {
  long long g = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

}  // namespace pfd

using namespace pfd;

extern "C" PFD_API int64_t pfd_canny_workspace_bytes(int32_t B, int32_t H, int32_t W) {
  const size_t px = (size_t)B * H * W;
  return (int64_t)(align256(px * 4) + align256(px * 4) + align256(px * 2) + align256(px) + 256);
}

extern "C" PFD_API int pfd_canny_f32(const void* x, int32_t src_is_f32, int32_t B, int32_t H, int32_t W,
                                     int32_t low, int32_t high, void* workspace, float* out,
                                     int32_t* sweeps_out, void* stream) {
  if (!x || !workspace || !out || B <= 0 || H <= 0 || W <= 0) return set_error("pfd_canny_f32: bad arguments");
  if (low > high) {
    const int32_t t = low;
    low = high;
    high = t;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t px = (size_t)B * H * W;
  char* ws = static_cast<char*>(workspace);
  uint32_t* rgbx = reinterpret_cast<uint32_t*>(ws);
  short2* dxy = reinterpret_cast<short2*>(ws + align256(px * 4));
  unsigned short* mag = reinterpret_cast<unsigned short*>(ws + align256(px * 4) * 2);
  unsigned char* map = reinterpret_cast<unsigned char*>(ws + align256(px * 4) * 2 + align256(px * 2));
  int* flag = reinterpret_cast<int*>(ws + align256(px * 4) * 2 + align256(px * 2) + align256(px));
  const int g = grid1d((long long)px);
  if (src_is_f32)
    launch_k(canny_pack_kernel<float>, dim3(g), dim3(256), (size_t)0, st, static_cast<const float*>(x), (int)B, (int)H, (int)W, rgbx);
  else
    launch_k(canny_pack_kernel<__half>, dim3(g), dim3(256), (size_t)0, st, static_cast<const __half*>(x), (int)B, (int)H, (int)W, rgbx);
  if (int rc = check_launch("canny_pack")) return rc;
  launch_k(canny_grad_kernel, dim3(g), dim3(256), (size_t)0, st, (const uint32_t*)rgbx, (int)B, (int)H, (int)W, dxy, mag);
  if (int rc = check_launch("canny_grad")) return rc;
  launch_k(canny_nms_kernel, dim3(g), dim3(256), (size_t)0, st, (const short2*)dxy, (const unsigned short*)mag, (int)B,
           (int)H, (int)W, (int)low, (int)high, map);
  if (int rc = check_launch("canny_nms")) return rc;
  // hysteresis sweeps until the fixed point (host-visible flag: this entry point synchronises the stream and is
  // therefore not capturable into a CUDA graph - it is request pre-processing, not part of the sampling loop)
  const dim3 hgrid((W + HT - 1) / HT, (H + HT - 1) / HT, B);
  int sweeps = 0;
  for (;;) {
    if (cudaMemsetAsync(flag, 0, sizeof(int), st) != cudaSuccess) return set_error("pfd_canny_f32: memset failed");
    launch_k(canny_hyst_kernel, hgrid, dim3(HT, HT), (size_t)0, st, map, (int)H, (int)W, flag);
    if (int rc = check_launch("canny_hyst")) return rc;
    int h_flag = 0;
    if (cudaMemcpyAsync(&h_flag, flag, sizeof(int), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
      return set_error("pfd_canny_f32: flag readback failed: %s", cudaGetErrorString(cudaGetLastError()));
    ++sweeps;
    if (!h_flag) break;
    if (sweeps > 65536) return set_error("pfd_canny_f32: hysteresis did not converge");
  }
  if (sweeps_out) *sweeps_out = sweeps;
  launch_k(canny_emit_kernel, dim3(g), dim3(256), (size_t)0, st, (const unsigned char*)map, (int)B, (int)H, (int)W, out);
  return check_launch("canny_emit");
}

extern "C" PFD_API int pfd_image_u8_roundtrip_f32(const void* x, int32_t src_is_f32, int64_t n, float* out,
                                                  void* stream) {
  if (!x || !out || n <= 0) return set_error("pfd_image_u8_roundtrip_f32: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (src_is_f32)
    launch_k(u8_roundtrip_kernel<float>, dim3(grid1d(n)), dim3(256), (size_t)0, st, static_cast<const float*>(x), (long long)n, out);
  else
    launch_k(u8_roundtrip_kernel<__half>, dim3(grid1d(n)), dim3(256), (size_t)0, st, static_cast<const __half*>(x), (long long)n, out);
  return check_launch("u8_roundtrip");
}
