// tcgen05 tensor-core contraction for sm_100a: one persistent, warp-specialised kernel that serves
// every Linear / 1x1 conv / 3x3 conv (implicit GEMM; TMA performs the im2col gather with
// zero-filled halos) / batched QK^T and PV product on the Prompt-Free-Diffusion hot path.
//
//   D[128 x BN] (fp32, TMEM)  +=  A[128 x 64] (fp16, smem, TMA 4-D box)  x  B[BN x 64]^T (fp16, smem)
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = tcgen05.mma issuer, warps 2..9 = epilogue
// (TMEM -> registers -> fused bias / time-embedding / activation / GEGLU / residual -> global).
// The accumulator is double-buffered in TMEM so the epilogue of tile i overlaps the main loop of
// tile i+1.  See include/pfd_b200.h (pfd_gemm_f16) for the reference call sites this replaces.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include <mutex>

#include "../../include/pfd_b200.h"
#include "common.h"
#include "ptx.cuh"

namespace pfd {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int UMMA_K = 16;
constexpr int GEMM_THREADS = 320;  // TMA warp, MMA warp, 8 epilogue warps
constexpr int STAGE_A_BYTES = BM * BK * 2;  // 16 KiB
constexpr int SMEM_BUDGET = 232448;         // 227 KiB opt-in limit per CTA
constexpr int EPI_WARPS = 8;
constexpr int EPI_STG_BYTES = 1024;         // per epilogue warp: 16 rows x 64 B transpose buffer
// TMA-store epilogue: every epilogue warp stages ITS share of the whole output tile (32 rows x up to ceil(BN/32)*16
// columns, fp16) so that the residual can be TMA-loaded into the same slabs while the main loop runs
constexpr int epi_stg_bytes(int bn, bool tmae) { return tmae ? 1024 * ((bn / 16 + 1) / 2) : EPI_STG_BYTES; }
// alignment slack + barriers + epilogue staging buffers + fp32 bias of the tile (double-buffered)
// (the TMA-store slabs must keep the 512-byte alignment of their swizzle pattern: the barrier block is padded to 1 KB)
constexpr int bar_block_bytes(bool tmae) { return tmae ? 1024 : 256; }
constexpr int smem_fixed(int bn, bool tmae) { return 1024 + bar_block_bytes(tmae) + EPI_WARPS * epi_stg_bytes(bn, tmae) + 2 * bn * 4; }

struct alignas(64) GemmParams {
  CUtensorMap tmA[PFD_MAX_SEG];
  CUtensorMap tmB;
  // TMA-store epilogue: output / residual rasters as 32-row slabs of 32 columns (SWIZZLE_64B) and 16 columns (SWIZZLE_32B)
  CUtensorMap tmO32, tmO16, tmR32, tmR16;
  int nseg;
  int taps[PFD_MAX_SEG];
  int chunks[PFD_MAX_SEG];
  int a_c[PFD_MAX_SEG];
  int stride;
  int tap_off;
  int bw, bh, bn;
  int tiles_w, tiles_h, tiles_nb, n_tiles;
  int W, H, NB, N;
  int b_batched;
  int num_kb;
  int splits;        // split-K factor (1 = off); work items = tiles * splits
  int kb_per_split;
  float* ws;         // fp32 partials [splits][m_tiles*128][N] when splits > 1
  // stream-K tail (single-CTA kernel, TMA-store epilogue): tiles < sk_dp_tiles are processed whole, one per CTA per
  // wave; the K blocks of the remaining sk_R tiles are spread evenly over ALL CTAs (see gemm_work)
  int sk_dp_tiles, sk_R;
  float* sk_ws;      // fp32 partial tiles [2 * grid][128][BN]
  int* sk_flags;     // [2 * grid] 0 / 1, reset by the consumer
  float alpha;
  int act;
  const __half* bias;
  const __half* rowadd;
  const __half* residual;
  __half* out;
  long long so_n1, so_n0, so_y, so_x, so_c1, so_c0;
  long long rowadd_ld;
  int ndiv, cdiv;
  int vec_ok;
};

template <int BN, bool TMAE = false>
struct GemmCfg {
  static constexpr int STAGE_B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = STAGE_A_BYTES + STAGE_B_BYTES;
  static constexpr int RAW_STAGES = (SMEM_BUDGET - smem_fixed(BN, TMAE)) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + smem_fixed(BN, TMAE);
  static constexpr int WARP_STG = epi_stg_bytes(BN, TMAE);
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128u : (2 * BN <= 256 ? 256u : 512u);
  static_assert(STAGE_B_BYTES % 1024 == 0, "B stage must keep 1024-B swizzle alignment");
  static_assert(BN % 16 == 0 && BN >= 16 && BN <= 256, "UMMA N constraint for M=128");
};

// erf to ~1.5e-7 absolute (Abramowitz & Stegun 7.1.26) with MUFU rcp/ex2: about half the
// instructions of erff(), far below the fp16 output resolution of the GELU / GEGLU epilogues.
__device__ __forceinline__ float fast_erf(float x) {
  const float ax = fabsf(x);
  const float t = __fdividef(1.f, fmaf(0.3275911f, ax, 1.f));
  float poly = fmaf(1.061405429f, t, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  const float y = 1.f - poly * __expf(-ax * ax);
  return copysignf(y, x);
}

// GELU as x * sigmoid(x * (a + b x^2 + c x^4)), coefficients fitted to the exact erf form on [-8, 8]
// (max |error| 2.5e-5, tools/fit_gelu.py; fp16 resolution near 1 is 4.9e-4).  The polynomial is evaluated on
// clamp(x, +-10) because c < 0 would flip its sign beyond |x| = 11.1; at |x| = 10 the sigmoid is already 0 / 1
// to 3e-9.  9 FMA-pipe instructions + 2 MUFU per element against ~17 + 2 for the A&S erf form.
__device__ __forceinline__ float gelu_sig(float x) {
  const float xc = fminf(fmaxf(x, -10.f), 10.f);
  const float x2 = xc * xc;
  // coefficients pre-multiplied by -log2(e)
  const float pl = fmaf(x2, fmaf(x2, 1.01426305e-3f, -1.06775723e-1f), -2.30112135f);
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(xc * pl));
  return __fdividef(x, 1.f + e);
}

// max(v, 0) that keeps NaN, as F.relu does: an fp16 overflow upstream (inf - inf = NaN) must reach the output
// instead of being flushed to 0
__device__ __forceinline__ float relu_nan(float v) {
  float r;
  asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(v));
  return r;
}

__device__ __forceinline__ float act_apply(float v, int act) {
  if (act == PFD_ACT_SILU) return __fdividef(v, 1.f + __expf(-v));
  if (act == PFD_ACT_GELU) return 0.5f * v * (1.f + fast_erf(v * 0.70710678118654752f));
  if (act == PFD_ACT_RELU) return relu_nan(v);
  return v;
}

__device__ __forceinline__ void unpack8h(const uint4& u, float (&f)[8]) {
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

__device__ __forceinline__ void load8h(const __half* p, float (&f)[8]) {
  uint4 u = __ldg(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __half22float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint4 hadd2x4(const uint4& a, const uint4& b) {
  uint4 o;
  const __half2* ah = reinterpret_cast<const __half2*>(&a);
  const __half2* bh = reinterpret_cast<const __half2*>(&b);
  __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
  for (int i = 0; i < 4; ++i) oh[i] = __hadd2(ah[i], bh[i]);
  return o;
}

__device__ __forceinline__ float4 ld_shared_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// One unit of work of a persistent CTA: K blocks [kb0, kb1) of output tile `tile`.
//   mode 0: the whole contraction of the tile (or, with split-K, slice `slot`) -> normal epilogue
//   mode 1: stream-K contributor: raw fp32 partial tile -> sk_ws[slot], then sk_flags[slot] = 1
//   mode 2: stream-K owner (its range ends with the tile's last K block): adds the contributors' partials, normal epilogue
// Stream-K tail: with T tiles on G CTAs the last wave holds R = T mod G tiles (every UNet conv: 0.46 or 0.73 or 0.86 of a
// wave, i.e. 13.5 % of the machine idle on average).  Their R * num_kb K blocks are cut into G equal contiguous ranges;
// a range covers the tail of one tile (processed LAST: this CTA owns that tile if it reaches its end) and possibly the
// head of the next (processed FIRST: a pure contributor that depends on nobody, so its partial is published early and
// the owner - the next CTA - rarely waits).
struct WorkItem {
  int tile, kb0, kb1, mode, slot;
};
__device__ __forceinline__ void sk_range(const GemmParams& p, int c, int G, int& u0, int& u1) {
  const long long U = (long long)p.sk_R * p.num_kb;
  u0 = (int)(U * c / G);
  u1 = (int)(U * (c + 1) / G);
}
template <bool SK>
__device__ __forceinline__ bool gemm_work(const GemmParams& p, int wi, int total_tiles, WorkItem& w) {
  const int G = gridDim.x, c = blockIdx.x;
  if (!SK || p.sk_R == 0) {
    const int work = c + wi * G;
    if (work >= total_tiles * p.splits) return false;
    w.tile = work % total_tiles;
    w.slot = work / total_tiles;
    w.kb0 = w.slot * p.kb_per_split;
    w.kb1 = min(p.num_kb, w.kb0 + p.kb_per_split);
    w.mode = 0;
    return true;
  }
  // The stream-K segments come FIRST and the whole tiles after them: the contributor -> flag -> owner hand-off
  // (MMA of the segment + partial store + release visibility + gather, ~10 us) is then hidden behind the whole
  // tiles of the same CTA (the accumulator is double-buffered, the MMA warp runs ahead of a waiting epilogue) and the
  // kernel ends with perfectly balanced whole tiles.  (Segments LAST measured 0.84-0.98x: the hand-off chain alone is
  // as long as a tile.)
  int u0, u1;
  sk_range(p, c, G, u0, u1);
  const int KB = p.num_kb;
  const int t0 = u0 / KB;
  const int aend = min(u1, (t0 + 1) * KB);
  const bool has_b = u1 > aend;                        // the range spills into tile t0 + 1
  const int nseg = (u1 > u0) ? (has_b ? 2 : 1) : 0;
  if (wi >= nseg) {
    const int n_dp = p.sk_dp_tiles / G;                // whole waves
    if (wi - nseg >= n_dp) return false;
    w.tile = c + (wi - nseg) * G; w.kb0 = 0; w.kb1 = p.num_kb; w.mode = 0; w.slot = 0;
    return true;
  }
  const int seg = wi;
  int s0, s1, t;
  if (seg == 0 && has_b) { s0 = aend; s1 = u1; t = t0 + 1; }
  else { s0 = u0; s1 = aend; t = t0; }
  w.tile = p.sk_dp_tiles + t;
  w.kb0 = s0 - t * KB;
  w.kb1 = s1 - t * KB;
  w.mode = (w.kb1 == KB) ? (w.kb0 == 0 ? 0 : 2) : 1;
  w.slot = 2 * c + ((seg == 0 && has_b) ? 1 : 0);
  return true;
}

// Per-warp view of one output tile for the TMA-store epilogue (shared by the single-CTA and the CTA-pair kernel).
struct EpiTile {
  int q, lane;                 // TMEM lane quarter / lane of the warp
  int tx, ty, tn;              // raster tile coordinates
  int cbeg, n32;               // first column of this warp inside the tile, number of 32-column runs
  bool tail16;                 // a 16-column tail run follows
  int col_base, n_lim;         // first output column of the tile, number of valid output columns
  bool has_res, valid;
  uint32_t stg, rbar, tfull, aph, taddr, sbias;
  float alpha;
  int act;
  const __half* rowadd_row;
  int sk_mode, sk_slot;        // stream-K: WorkItem::mode / slot (0 / unused for whole tiles)
  int sk_t, sk_kb0;            // stream-K owner: index of the tile in the tail, first K block of its own range
  int stg_warp;                // index of this epilogue warp (0..7)
};

__device__ __forceinline__ int ld_acquire_gpu(const int* ptr) {
  int v;
  asm volatile("ld.acquire.gpu.global.b32 %0, [%1];" : "=r"(v) : "l"(ptr) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(int* ptr, int v) {
  asm volatile("st.release.gpu.global.b32 [%0], %1;" ::"l"(ptr), "r"(v) : "memory");
}

// ---------------- TMA-store epilogue.  This warp owns rows [32q, 32q+32) x columns [cbeg, cend) of the tile
// and a private staging area holding that share as slabs of 32 rows x 32 columns (2 KB, SWIZZLE_64B) plus at
// most one 16-column tail slab (1 KB, SWIZZLE_32B).  Per tile: (1) wait until the previous tile's stores have
// read the staging area, (2) one lane TMA-loads the residual slabs into it (arrives while the main loop of
// this tile is still running), (3) per slab: tcgen05.ld -> bias / row add / activation in fp32 -> fp16 ->
// fp16 add of the residual read back from the slab (the reference's `x + f(h)` on fp16 tensors) -> in-place
// st.shared (conflict-free in the swizzled layout) -> fence.proxy.async -> one lane issues the TMA store.
// Out-of-raster rows and columns >= N are clipped by the TMA unit, so there is no per-row predicate, no
// 64-bit address arithmetic and no global load/store instruction left in the loop.
template <int BN, bool SK>
__device__ __forceinline__ void tma_store_epilogue(const GemmParams& p, const EpiTile& e, uint32_t& res_phase) {
  const int q = e.q, lane = e.lane, tx = e.tx, ty = e.ty, tn = e.tn, cbeg = e.cbeg, n32 = e.n32;
  const bool tail16 = e.tail16, has_res = e.has_res, valid = e.valid;
  const int col_base = e.col_base, n_lim = e.n_lim, act = e.act;
  const uint32_t stg = e.stg, taddr = e.taddr, sbias = e.sbias;
  const float alpha = e.alpha;
  const __half* rowadd_row = e.rowadd_row;
  const int r0 = q * 32;
  const int gx = tx * p.bw + r0 % p.bw;
  const int gy = ty * p.bh + (r0 / p.bw) % p.bh;
  const int gn = tn * p.bn + r0 / (p.bw * p.bh);
  int live32 = 0;
  for (int i = 0; i < n32; ++i) live32 += (col_base + cbeg + 32 * i < n_lim) ? 1 : 0;
  const bool live16 = tail16 && (col_base + cbeg + 32 * n32 < n_lim);
  const uint32_t rb_addr = e.rbar;
  if (SK && e.sk_mode == 1) {
    // ---- stream-K contributor: raw fp32 accumulators of this CTA's K range -> sk_ws[slot][row][col], then publish
    // partial-tile layout: private to the (contributor warp, owner warp) pair that share a tile position, so it is chosen
    // for the memory system, not for humans: [slot][warp][16-byte group g of the warp's columns][lane] -> every
    // warp-wide store / load is one contiguous 512-byte request (the row-major version cost 6 + 12 us per tile)
    uint4* pw = reinterpret_cast<uint4*>(p.sk_ws) + ((long long)e.sk_slot * EPI_WARPS + (e.stg_warp)) * (BN / 8) * 32 + lane;
    mbar_wait(e.tfull, e.aph);
    tc_fence_after();
    for (int i = 0; i < live32; ++i) {
      const int c0 = cbeg + 32 * i;
      uint32_t r[32];
      tmem_ld32(taddr + c0, r);
      tmem_ld_wait();
#pragma unroll
      for (int v4 = 0; v4 < 8; ++v4)
        __stcg(pw + (i * 8 + v4) * 32, make_uint4(r[4 * v4], r[4 * v4 + 1], r[4 * v4 + 2], r[4 * v4 + 3]));
    }
    if (live16) {
      const int c0 = cbeg + 32 * n32;
      uint32_t r[16];
      tmem_ld16(taddr + c0, r);
      tmem_ld_wait();
#pragma unroll
      for (int v4 = 0; v4 < 4; ++v4)
        __stcg(pw + (n32 * 8 + v4) * 32, make_uint4(r[4 * v4], r[4 * v4 + 1], r[4 * v4 + 2], r[4 * v4 + 3]));
    }
    __threadfence();
    asm volatile("bar.sync 1, 256;" ::: "memory");          // every epilogue thread's partial rows are written and fenced
    if (threadIdx.x == 64) st_release_gpu(p.sk_flags + e.sk_slot, 1);
    return;
  }
  // stream-K owner: the CTAs whose ranges cover K blocks [0, sk_kb0) of this tile; their partial tiles are added to the
  // accumulator before the normal epilogue.  Contributor cc used slot 2cc if its range STARTS inside this tile
  // (its tail part) and slot 2cc + 1 if it spilled over from the previous tile (its head part).
  int nsrc = 0, src_slot[6];
  if (SK && e.sk_mode == 2) {
    const int G = gridDim.x;
    const int tstart = e.sk_t * p.num_kb;
    for (int cc = (int)blockIdx.x - 1; cc >= 0 && nsrc < 6; --cc) {
      int u0, u1;
      sk_range(p, cc, G, u0, u1);
      if (u1 <= tstart) break;
      if (u1 > u0) src_slot[nsrc++] = (u0 >= tstart) ? 2 * cc : 2 * cc + 1;
    }
    if (threadIdx.x == 64) {
      for (int j = 0; j < nsrc; ++j) {
        uint32_t spins = 0;
        while (ld_acquire_gpu(p.sk_flags + src_slot[j]) == 0) {
          __nanosleep(64);
          if (++spins > (1u << 24)) asm volatile("trap;");
        }
        p.sk_flags[src_slot[j]] = 0;                       // consumed: ready for the next launch
      }
    }
  }
  if (lane == 0) {
    bulk_wait_read_all();                         // stores of the previous tile have read the slabs
    if (has_res && (live32 > 0 || live16)) {
      mbar_expect_tx(rb_addr, live32 * 2048 + (live16 ? 1024 : 0));
      for (int i = 0; i < live32; ++i)
        tma_load_4d(stg + i * 2048, &p.tmR32, rb_addr, col_base + cbeg + 32 * i, gx, gy, gn);
      if (live16) tma_load_4d(stg + n32 * 2048, &p.tmR16, rb_addr, col_base + cbeg + 32 * n32, gx, gy, gn);
    }
  }
  __syncwarp();
  asm volatile("bar.sync 1, 256;" ::: "memory");          // bias of this tile visible to all epilogue warps
  mbar_wait(e.tfull, e.aph);
  tc_fence_after();
  if (has_res && (live32 > 0 || live16)) {
    mbar_wait(rb_addr, res_phase);
    res_phase ^= 1u;
  }
  const uint32_t sw64 = (lane >> 1) & 3, sw32 = (lane >> 2) & 1;
  for (int i = 0; i < live32; ++i) {
    const int c0 = cbeg + 32 * i;
    uint32_t r[32];
    tmem_ld32(taddr + c0, r);
    tmem_ld_wait();
    for (int j = 0; SK && j < nsrc; ++j) {
      const uint4* src = reinterpret_cast<const uint4*>(p.sk_ws) +
                         (((long long)src_slot[j] * EPI_WARPS + e.stg_warp) * (BN / 8) + i * 8) * 32 + lane;
#pragma unroll
      for (int v4 = 0; v4 < 8; ++v4) {
        const uint4 u = __ldcg(src + v4 * 32);
        r[4 * v4] = __float_as_uint(__uint_as_float(r[4 * v4]) + __uint_as_float(u.x));
        r[4 * v4 + 1] = __float_as_uint(__uint_as_float(r[4 * v4 + 1]) + __uint_as_float(u.y));
        r[4 * v4 + 2] = __float_as_uint(__uint_as_float(r[4 * v4 + 2]) + __uint_as_float(u.z));
        r[4 * v4 + 3] = __float_as_uint(__uint_as_float(r[4 * v4 + 3]) + __uint_as_float(u.w));
      }
    }
    uint32_t h[16];
    if (rowadd_row == nullptr && act == PFD_ACT_NONE) {
#pragma unroll
      for (int q4 = 0; q4 < 8; ++q4) {
        const float4 b = ld_shared_f4(sbias + (c0 + q4 * 4) * 4);
        h[q4 * 2] = pack_h2(fmaf(__uint_as_float(r[q4 * 4]), alpha, b.x), fmaf(__uint_as_float(r[q4 * 4 + 1]), alpha, b.y));
        h[q4 * 2 + 1] = pack_h2(fmaf(__uint_as_float(r[q4 * 4 + 2]), alpha, b.z), fmaf(__uint_as_float(r[q4 * 4 + 3]), alpha, b.w));
      }
    } else {
#pragma unroll
      for (int q8 = 0; q8 < 4; ++q8) {
        float v[8];
        const float4 b0 = ld_shared_f4(sbias + (c0 + q8 * 8) * 4);
        const float4 b1 = ld_shared_f4(sbias + (c0 + q8 * 8 + 4) * 4);
        v[0] = fmaf(__uint_as_float(r[q8 * 8]), alpha, b0.x);
        v[1] = fmaf(__uint_as_float(r[q8 * 8 + 1]), alpha, b0.y);
        v[2] = fmaf(__uint_as_float(r[q8 * 8 + 2]), alpha, b0.z);
        v[3] = fmaf(__uint_as_float(r[q8 * 8 + 3]), alpha, b0.w);
        v[4] = fmaf(__uint_as_float(r[q8 * 8 + 4]), alpha, b1.x);
        v[5] = fmaf(__uint_as_float(r[q8 * 8 + 5]), alpha, b1.y);
        v[6] = fmaf(__uint_as_float(r[q8 * 8 + 6]), alpha, b1.z);
        v[7] = fmaf(__uint_as_float(r[q8 * 8 + 7]), alpha, b1.w);
        if (rowadd_row != nullptr && valid && col_base + c0 + q8 * 8 < n_lim) {
          float rv[8];
          load8h(rowadd_row + col_base + c0 + q8 * 8, rv);
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] += rv[k];
        }
        if (act != PFD_ACT_NONE) {
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = act_apply(v[k], act);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) h[q8 * 4 + k] = pack_h2(v[2 * k], v[2 * k + 1]);
      }
    }
    const uint32_t slab = stg + i * 2048 + lane * 64;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t a = slab + ((k ^ sw64) << 4);
      uint4 o = make_uint4(h[4 * k], h[4 * k + 1], h[4 * k + 2], h[4 * k + 3]);
      if (has_res) o = hadd2x4(o, ld_shared_v4(a));
      st_shared_v4(a, o.x, o.y, o.z, o.w);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) tma_store_4d(&p.tmO32, stg + i * 2048, col_base + c0, gx, gy, gn);
  }
  if (live16) {
    const int c0 = cbeg + 32 * n32;
    uint32_t r[16];
    tmem_ld16(taddr + c0, r);
    tmem_ld_wait();
    for (int j = 0; SK && j < nsrc; ++j) {
      const uint4* src = reinterpret_cast<const uint4*>(p.sk_ws) +
                         (((long long)src_slot[j] * EPI_WARPS + e.stg_warp) * (BN / 8) + n32 * 8) * 32 + lane;
#pragma unroll
      for (int v4 = 0; v4 < 4; ++v4) {
        const uint4 u = __ldcg(src + v4 * 32);
        r[4 * v4] = __float_as_uint(__uint_as_float(r[4 * v4]) + __uint_as_float(u.x));
        r[4 * v4 + 1] = __float_as_uint(__uint_as_float(r[4 * v4 + 1]) + __uint_as_float(u.y));
        r[4 * v4 + 2] = __float_as_uint(__uint_as_float(r[4 * v4 + 2]) + __uint_as_float(u.z));
        r[4 * v4 + 3] = __float_as_uint(__uint_as_float(r[4 * v4 + 3]) + __uint_as_float(u.w));
      }
    }
    uint32_t h[8];
#pragma unroll
    for (int q8 = 0; q8 < 2; ++q8) {
      float v[8];
      const float4 b0 = ld_shared_f4(sbias + (c0 + q8 * 8) * 4);
      const float4 b1 = ld_shared_f4(sbias + (c0 + q8 * 8 + 4) * 4);
      v[0] = fmaf(__uint_as_float(r[q8 * 8]), alpha, b0.x);
      v[1] = fmaf(__uint_as_float(r[q8 * 8 + 1]), alpha, b0.y);
      v[2] = fmaf(__uint_as_float(r[q8 * 8 + 2]), alpha, b0.z);
      v[3] = fmaf(__uint_as_float(r[q8 * 8 + 3]), alpha, b0.w);
      v[4] = fmaf(__uint_as_float(r[q8 * 8 + 4]), alpha, b1.x);
      v[5] = fmaf(__uint_as_float(r[q8 * 8 + 5]), alpha, b1.y);
      v[6] = fmaf(__uint_as_float(r[q8 * 8 + 6]), alpha, b1.z);
      v[7] = fmaf(__uint_as_float(r[q8 * 8 + 7]), alpha, b1.w);
      if (rowadd_row != nullptr && valid && col_base + c0 + q8 * 8 < n_lim) {
        float rv[8];
        load8h(rowadd_row + col_base + c0 + q8 * 8, rv);
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] += rv[k];
      }
      if (act != PFD_ACT_NONE) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = act_apply(v[k], act);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) h[q8 * 4 + k] = pack_h2(v[2 * k], v[2 * k + 1]);
    }
    const uint32_t slab = stg + n32 * 2048 + lane * 32;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const uint32_t a = slab + ((k ^ sw32) << 4);
      uint4 o = make_uint4(h[4 * k], h[4 * k + 1], h[4 * k + 2], h[4 * k + 3]);
      if (has_res) o = hadd2x4(o, ld_shared_v4(a));
      st_shared_v4(a, o.x, o.y, o.z, o.w);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) tma_store_4d(&p.tmO16, stg + n32 * 2048, col_base + c0, gx, gy, gn);
  }
  if (lane == 0) bulk_commit_group();
}

// LEAN = true: epilogue for 16-byte-vectorisable outputs (channel-last rows, optional head split) without split-K;
// LEAN = false keeps the general path (element-strided outputs such as V^T, split-K partials).
// TMAE = true (implies LEAN, plain channel-last output, no GEGLU / split-K): the tile leaves through TMA stores and the
// residual arrives through TMA loads (see the epilogue).
// SK = true (implies TMAE): stream-K tail enabled (gemm_work / epilogue modes); a separate instantiation because the extra
// epilogue state costs the plain kernel 2.5 % (152 vs 140 registers + the work-item arithmetic in all three roles).
template <int BN, bool LEAN, bool TMAE, bool SK>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BN, TMAE>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];

  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - raw_addr);
  const uint32_t smemA = base;
  const uint32_t smemB = base + STAGES * STAGE_A_BYTES;               // [STAGES][B tile]
  constexpr int nst = STAGES;
  const uint32_t bars = base + STAGES * Cfg::STAGE_BYTES;
  // barrier layout: full[STAGES] | empty[STAGES] | tmem_full[2] | tmem_empty[2] | tmem_ptr
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * STAGES + 4);
  auto res_bar = [&](int w) { return bars + 8u * (2 * STAGES + 5 + w); };    // one per epilogue warp (TMAE)
  volatile uint32_t* tmem_slot_g =
      reinterpret_cast<volatile uint32_t*>(gbase + STAGES * Cfg::STAGE_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nseg; ++s) tma_prefetch_desc(&p.tmA[s]);
    tma_prefetch_desc(&p.tmB);
    if (TMAE) {
      tma_prefetch_desc(&p.tmO32);
      tma_prefetch_desc(&p.tmO16);
      if (p.residual) {
        tma_prefetch_desc(&p.tmR32);
        tma_prefetch_desc(&p.tmR16);
      }
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 256);
    }
    if (TMAE)
      for (int w = 0; w < EPI_WARPS; ++w) mbar_init(res_bar(w), 1);
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_g;
  // prologue above overlapped the previous kernel's tail; global data may only be touched from here on
  pdl_wait();
  pdl_launch_dependents();

  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_nb;
  const int total_tiles = m_tiles * p.n_tiles;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      WorkItem w;
      for (int wi = 0; gemm_work<SK>(p, wi, total_tiles, w); ++wi) {
        const int tile = w.tile;
        const int kb_begin = w.kb0, kb_end = w.kb1;
        const int n_tile = tile % p.n_tiles;
        const int m_tile = tile / p.n_tiles;
        const int tx = m_tile % p.tiles_w;
        const int ty = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const int x0 = tx * p.bw * p.stride;
        const int y0 = ty * p.bh * p.stride;
        const int n0 = tn * p.bn;
        const int bcoord = p.b_batched ? n0 : 0;
        int kofs = 0;
        int kbi = 0;
        for (int s = 0; s < p.nseg; ++s) {
          const int ntap = p.taps[s];
          for (int t = 0; t < ntap; ++t) {
            const int dy = (ntap == 9) ? (t / 3 - 1 + p.tap_off) : 0;
            const int dx = (ntap == 9) ? (t % 3 - 1 + p.tap_off) : 0;
            for (int j = 0; j < p.chunks[s]; ++j, ++kbi) {
              if (kbi < kb_begin || kbi >= kb_end) continue;
              mbar_wait(empty_bar(stage), phase ^ 1u);
              mbar_expect_tx(full_bar(stage), Cfg::STAGE_BYTES);
              tma_load_4d(smemA + stage * STAGE_A_BYTES, &p.tmA[s], full_bar(stage), j * BK,
                          x0 + dx, y0 + dy, n0);
              tma_load_3d(smemB + stage * Cfg::STAGE_B_BYTES, &p.tmB, full_bar(stage),
                          kofs + j * BK, n_tile * BN, bcoord);
              if (++stage == nst) {
                stage = 0;
                phase ^= 1u;
              }
            }
            kofs += p.a_c[s];
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (one thread)
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_f16(BN);
      int stage = 0;
      uint32_t phase = 0;
      WorkItem w;
      for (int it = 0; gemm_work<SK>(p, it, total_tiles, w); ++it) {
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        const int nkb = w.kb1 - w.kb0;
        mbar_wait(tempty_bar(as), aph ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint64_t adesc = make_sw128_kmajor_desc(smemA + stage * STAGE_A_BYTES);
          const uint64_t bdesc = make_sw128_kmajor_desc(smemB + stage * Cfg::STAGE_B_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            // advance 16 fp16 = 32 B inside the 128-B swizzle atom: +2 in the (addr>>4) field
            umma_f16(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          umma_commit(empty_bar(stage));
          if (++stage == nst) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(tfull_bar(as));
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 2..9)
    // Two warps per TMEM lane quarter, each owning half of the tile's column chunks: the lone-warp-per-
    // scheduler epilogue was latency-bound (ncu: 214 instr and several exposed load latencies per
    // 16 columns).  Per chunk all global loads (bias / row add / residual) are issued before the
    // TMEM load is waited on, index arithmetic is hoisted out of the chunk loop.
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int half_id = (warp - 2) >> 2;    // 0: warps 2..5, 1: warps 6..9
    const int row = q * 32 + lane;
    const int rdx = row % p.bw;
    const int rdy = (row / p.bw) % p.bh;
    const int rdn = row / (p.bw * p.bh);
    const bool geglu = (p.act == PFD_ACT_GEGLU);
    const int n_out = geglu ? p.N / 2 : p.N;
    constexpr int CB = BN;                  // accumulator columns per tile in TMEM
    const int ocols = geglu ? CB / 2 : CB;  // output columns this tile produces
    const int nch = ocols / 16;
    const int ch_begin = half_id == 0 ? 0 : (nch + 1) / 2;
    const int ch_end = half_id == 0 ? (nch + 1) / 2 : nch;
    const bool plain_cols = p.cdiv >= p.N;  // no head split: column offset = col * so_c0
    uint32_t res_phase = 0;                 // TMAE: parity of this warp's residual barrier
    WorkItem w;
    for (int it = 0; gemm_work<SK>(p, it, total_tiles, w); ++it) {
      const int tile = w.tile;
      const int split = w.slot;
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int n_tile = tile % p.n_tiles;
      const int m_tile = tile / p.n_tiles;
      const int tx = m_tile % p.tiles_w;
      const int ty = (m_tile / p.tiles_w) % p.tiles_h;
      const int tn = m_tile / (p.tiles_w * p.tiles_h);
      const int x = tx * p.bw + rdx;
      const int y = ty * p.bh + rdy;
      const int n = tn * p.bn + rdn;
      const bool valid = (x < p.W) && (y < p.H) && (n < p.NB);
      const long long row_off = (long long)(n / p.ndiv) * p.so_n1 + (long long)(n % p.ndiv) * p.so_n0 +
                                (long long)y * p.so_y + (long long)x * p.so_x;
      const int col_base = n_tile * ocols;  // first output column of the tile
      const __half* rowadd_row = p.rowadd ? p.rowadd + (long long)n * p.rowadd_ld : nullptr;
      // (head, element) of the first column this warp handles, advanced by 8 per half-chunk
      int hcol = 0, ecol = col_base + ch_begin * 16;
      if (!plain_cols) {
        hcol = ecol / p.cdiv;
        ecol = ecol % p.cdiv;
      }
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * CB;
      if constexpr (LEAN) {
        // ---------------- lean path (r1 ncu prof_lin: the general epilogue issued ~270 instructions per 16
        // columns at ~8 cycles each with 2 warps per scheduler, and every row-per-thread ld/st.global request
        // touched 32 lines -> small-K GEMMs spent 2.7-5.2 us per tile here against 0.8 us of MMA).
        //  * the tile's bias is converted to fp32 once into shared memory (double-buffered by accumulator
        //    stage, one named barrier per tile) -> one FFMA per element (acc * alpha + bias);
        //  * runs of 32 columns: tcgen05.ld 32 columns, pack to fp16, transpose the warp's 32 rows x 64 B
        //    through a 1 KB XOR-swizzled buffer (two half-warp passes, conflict-free both ways) so that
        //    global traffic is 8 rows x 64 B per request;
        //  * the residual is read in the same coalesced mapping, one run ahead (run 0: before the
        //    accumulator is ready), and added to the fp16-rounded result in fp16 - the reference's
        //    `x + conv(h)` on fp16 tensors.
        const uint32_t fixed0 = base + STAGES * Cfg::STAGE_BYTES + bar_block_bytes(TMAE);
        const uint32_t stg = fixed0 + (warp - 2) * Cfg::WARP_STG;
        const uint32_t sbias = fixed0 + EPI_WARPS * Cfg::WARP_STG + as * (BN * 4);
        const int et = threadIdx.x - 64;
        if (et < BN) {
          // GEGLU weights/bias are packed [value | gate] per n tile (pack_geglu): bias index n_tile * BN + j
          const int c = geglu ? n_tile * BN + et : col_base + et;
          const float b = (p.bias != nullptr && c < p.N) ? __half2float(__ldg(p.bias + c)) : 0.f;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(sbias + et * 4), "f"(b) : "memory");
        }
        const int cbeg = ch_begin * 16, cend = ch_end * 16;        // this warp's columns inside the tile
        const int n32 = (cend - cbeg) >> 5;
        const bool tail16 = ((cend - cbeg) & 16) != 0;
        const long long my_off = valid ? row_off : -1;
        // 32-column runs: 4 lanes per row, rows hp*16 + it*8 + lane/4; 16-column run: 2 lanes per row, rows it*16 + lane/2
        const int cc4 = lane & 3, cc2 = lane & 1;
        long long roff4[4], roff2[2];
#pragma unroll
        for (int j = 0; j < 4; ++j) roff4[j] = __shfl_sync(0xffffffffu, my_off, (j >> 1) * 16 + (j & 1) * 8 + (lane >> 2));
#pragma unroll
        for (int j = 0; j < 2; ++j) roff2[j] = __shfl_sync(0xffffffffu, my_off, j * 16 + (lane >> 1));
        const __half* resp = p.residual;
        const bool has_res = resp != nullptr;
        const float alpha = p.alpha;
        const int act = p.act;
        const int n_lim = n_out;
        // element offset of output column c: head split (c / cdiv) * so_c1 + c % cdiv, or just c
        auto coff_of = [&](int c) -> long long {
          return plain_cols ? (long long)c : (long long)(c / p.cdiv) * p.so_c1 + (long long)(c % p.cdiv);
        };
        auto load_res32 = [&](int c0, uint4(&dst)[4]) {
          const int c = col_base + c0 + cc4 * 8;
          if (has_res && c < n_lim) {
            const long long co = coff_of(c);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (roff4[j] >= 0) dst[j] = __ldg(reinterpret_cast<const uint4*>(resp + roff4[j] + co));
          }
        };
        auto load_res16 = [&](int c0, uint4(&dst)[4]) {
          const int c = col_base + c0 + cc2 * 8;
          if (has_res && c < n_lim) {
            const long long co = coff_of(c);
#pragma unroll
            for (int j = 0; j < 2; ++j)
              if (roff2[j] >= 0) dst[j] = __ldg(reinterpret_cast<const uint4*>(resp + roff2[j] + co));
          }
        };
        if (geglu) {
          // ------ GEGLU: out[:, col] = value * gelu(gate), runs of 16 output columns (value + gate accumulators)
          asm volatile("bar.sync 1, 256;" ::: "memory");
          mbar_wait(tfull_bar(as), aph);
          tc_fence_after();
          const uint32_t wr16 = stg + lane * 32;
          const uint32_t swz16 = (lane >> 2) & 1;
          for (int ch = ch_begin; ch < ch_end; ++ch) {
            const int c0 = ch * 16;
            uint32_t r[16], g[16];
            tmem_ld16(taddr + c0, r);
            tmem_ld16(taddr + CB / 2 + c0, g);
            tmem_ld_wait();
            uint32_t h[8];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const float4 b = ld_shared_f4(sbias + (c0 + q4 * 4) * 4);
              const float4 bg = ld_shared_f4(sbias + (CB / 2 + c0 + q4 * 4) * 4);
              // reference: x, gate = proj(x).chunk(2) are fp16 tensors; x * gelu(gate) in fp16 (attention.py:50-51)
              const __half2 a01 = __floats2half2_rn(fmaf(__uint_as_float(r[q4 * 4]), alpha, b.x), fmaf(__uint_as_float(r[q4 * 4 + 1]), alpha, b.y));
              const __half2 a23 = __floats2half2_rn(fmaf(__uint_as_float(r[q4 * 4 + 2]), alpha, b.z), fmaf(__uint_as_float(r[q4 * 4 + 3]), alpha, b.w));
              const float2 g01 = __half22float2(__floats2half2_rn(fmaf(__uint_as_float(g[q4 * 4]), alpha, bg.x), fmaf(__uint_as_float(g[q4 * 4 + 1]), alpha, bg.y)));
              const float2 g23 = __half22float2(__floats2half2_rn(fmaf(__uint_as_float(g[q4 * 4 + 2]), alpha, bg.z), fmaf(__uint_as_float(g[q4 * 4 + 3]), alpha, bg.w)));
              const __half2 o01 = __hmul2(a01, __floats2half2_rn(gelu_sig(g01.x), gelu_sig(g01.y)));
              const __half2 o23 = __hmul2(a23, __floats2half2_rn(gelu_sig(g23.x), gelu_sig(g23.y)));
              h[q4 * 2] = *reinterpret_cast<const uint32_t*>(&o01);
              h[q4 * 2 + 1] = *reinterpret_cast<const uint32_t*>(&o23);
            }
            st_shared_v4(wr16 + ((0 ^ swz16) << 4), h[0], h[1], h[2], h[3]);
            st_shared_v4(wr16 + ((1 ^ swz16) << 4), h[4], h[5], h[6], h[7]);
            __syncwarp();
            const int c = col_base + c0 + cc2 * 8;
#pragma unroll
            for (int it = 0; it < 2; ++it) {
              const int rr = it * 16 + (lane >> 1);
              if (roff2[it] >= 0) {
                const uint4 o = ld_shared_v4(stg + rr * 32 + ((cc2 ^ ((rr >> 2) & 1)) << 4));
                *reinterpret_cast<uint4*>(p.out + roff2[it] + c) = o;
              }
            }
            __syncwarp();
          }
          tc_fence_before();
          mbar_arrive(tempty_bar(as));
          continue;
        }
        if constexpr (TMAE) {
          EpiTile e;
          e.q = q; e.lane = lane; e.tx = tx; e.ty = ty; e.tn = tn; e.cbeg = cbeg; e.n32 = n32; e.tail16 = tail16;
          e.col_base = col_base; e.n_lim = n_lim; e.has_res = has_res; e.valid = valid;
          e.stg = stg; e.rbar = res_bar(warp - 2); e.tfull = tfull_bar(as); e.aph = aph; e.taddr = taddr; e.sbias = sbias;
          e.alpha = alpha; e.act = act; e.rowadd_row = rowadd_row;
          e.sk_mode = w.mode; e.sk_slot = w.slot; e.sk_t = w.tile - p.sk_dp_tiles; e.sk_kb0 = w.kb0; e.stg_warp = warp - 2;
          tma_store_epilogue<BN, SK>(p, e, res_phase);
          tc_fence_before();
          mbar_arrive(tempty_bar(as));
          continue;
        }
        uint4 ra[4], rb[4];
        int c0 = cbeg;
        if (n32 > 0) load_res32(c0, ra);
        else if (tail16) load_res16(c0, ra);
        asm volatile("bar.sync 1, 256;" ::: "memory");            // bias of this tile visible to all epilogue warps
        mbar_wait(tfull_bar(as), aph);
        tc_fence_after();
        const uint32_t wr32 = stg + (lane & 15) * 64;
        const uint32_t swz32 = ((lane & 15) >> 1) & 3;
        const uint32_t rd32 = stg + (lane >> 2) * 64 + ((cc4 ^ ((lane >> 3) & 3)) << 4);
        for (int i = 0; i < n32; ++i, c0 += 32) {
          if (col_base + c0 >= n_lim) break;                       // warp-uniform
          uint32_t r[32];
          tmem_ld32(taddr + c0, r);
          if (i + 1 < n32) load_res32(c0 + 32, rb);
          else if (tail16) load_res16(c0 + 32, rb);
          tmem_ld_wait();
          uint32_t h[16];
          if (rowadd_row == nullptr && act == PFD_ACT_NONE) {
#pragma unroll
            for (int q4 = 0; q4 < 8; ++q4) {
              const float4 b = ld_shared_f4(sbias + (c0 + q4 * 4) * 4);
              h[q4 * 2] = pack_h2(fmaf(__uint_as_float(r[q4 * 4]), alpha, b.x), fmaf(__uint_as_float(r[q4 * 4 + 1]), alpha, b.y));
              h[q4 * 2 + 1] = pack_h2(fmaf(__uint_as_float(r[q4 * 4 + 2]), alpha, b.z), fmaf(__uint_as_float(r[q4 * 4 + 3]), alpha, b.w));
            }
          } else {
            // per-image row add (time embedding) and/or activation: same order as the reference
            // (conv + bias) + emb -> act
#pragma unroll
            for (int q8 = 0; q8 < 4; ++q8) {
              float v[8];
              const float4 b0 = ld_shared_f4(sbias + (c0 + q8 * 8) * 4);
              const float4 b1 = ld_shared_f4(sbias + (c0 + q8 * 8 + 4) * 4);
              v[0] = fmaf(__uint_as_float(r[q8 * 8]), alpha, b0.x);
              v[1] = fmaf(__uint_as_float(r[q8 * 8 + 1]), alpha, b0.y);
              v[2] = fmaf(__uint_as_float(r[q8 * 8 + 2]), alpha, b0.z);
              v[3] = fmaf(__uint_as_float(r[q8 * 8 + 3]), alpha, b0.w);
              v[4] = fmaf(__uint_as_float(r[q8 * 8 + 4]), alpha, b1.x);
              v[5] = fmaf(__uint_as_float(r[q8 * 8 + 5]), alpha, b1.y);
              v[6] = fmaf(__uint_as_float(r[q8 * 8 + 6]), alpha, b1.z);
              v[7] = fmaf(__uint_as_float(r[q8 * 8 + 7]), alpha, b1.w);
              if (rowadd_row != nullptr && valid && col_base + c0 + q8 * 8 < n_lim) {
                float rv[8];
                load8h(rowadd_row + col_base + c0 + q8 * 8, rv);
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += rv[i];
              }
              if (act != PFD_ACT_NONE) {
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = act_apply(v[i], act);
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) h[q8 * 4 + i] = pack_h2(v[2 * i], v[2 * i + 1]);
            }
          }
          const int c = col_base + c0 + cc4 * 8;
          const bool colok = c < n_lim;
          const long long co = coff_of(c);
#pragma unroll
          for (int hp = 0; hp < 2; ++hp) {
            if ((lane >> 4) == hp) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                st_shared_v4(wr32 + ((k ^ swz32) << 4), h[4 * k], h[4 * k + 1], h[4 * k + 2], h[4 * k + 3]);
            }
            __syncwarp();
#pragma unroll
            for (int it = 0; it < 2; ++it) {
              const int j = hp * 2 + it;
              if (colok && roff4[j] >= 0) {
                uint4 o = ld_shared_v4(rd32 + it * 512);
                if (has_res) o = hadd2x4(o, ra[j]);
                *reinterpret_cast<uint4*>(p.out + roff4[j] + co) = o;
              }
            }
            __syncwarp();
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) ra[j] = rb[j];
        }
        if (tail16 && col_base + c0 < n_lim) {
          uint32_t r[16];
          tmem_ld16(taddr + c0, r);
          tmem_ld_wait();
          uint32_t h[8];
#pragma unroll
          for (int q8 = 0; q8 < 2; ++q8) {
            float v[8];
            const float4 b0 = ld_shared_f4(sbias + (c0 + q8 * 8) * 4);
            const float4 b1 = ld_shared_f4(sbias + (c0 + q8 * 8 + 4) * 4);
            v[0] = fmaf(__uint_as_float(r[q8 * 8]), alpha, b0.x);
            v[1] = fmaf(__uint_as_float(r[q8 * 8 + 1]), alpha, b0.y);
            v[2] = fmaf(__uint_as_float(r[q8 * 8 + 2]), alpha, b0.z);
            v[3] = fmaf(__uint_as_float(r[q8 * 8 + 3]), alpha, b0.w);
            v[4] = fmaf(__uint_as_float(r[q8 * 8 + 4]), alpha, b1.x);
            v[5] = fmaf(__uint_as_float(r[q8 * 8 + 5]), alpha, b1.y);
            v[6] = fmaf(__uint_as_float(r[q8 * 8 + 6]), alpha, b1.z);
            v[7] = fmaf(__uint_as_float(r[q8 * 8 + 7]), alpha, b1.w);
            if (rowadd_row != nullptr && valid && col_base + c0 + q8 * 8 < n_lim) {
              float rv[8];
              load8h(rowadd_row + col_base + c0 + q8 * 8, rv);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] += rv[i];
            }
            if (act != PFD_ACT_NONE) {
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = act_apply(v[i], act);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) h[q8 * 4 + i] = pack_h2(v[2 * i], v[2 * i + 1]);
          }
          // 32 rows x 32 B in one pass: chunk k of row l at l*32 + ((k ^ ((l >> 2) & 1)) << 4)
          const uint32_t wr16 = stg + lane * 32;
          const uint32_t swz16 = (lane >> 2) & 1;
          st_shared_v4(wr16 + ((0 ^ swz16) << 4), h[0], h[1], h[2], h[3]);
          st_shared_v4(wr16 + ((1 ^ swz16) << 4), h[4], h[5], h[6], h[7]);
          __syncwarp();
          const int c = col_base + c0 + cc2 * 8;
          if (c < n_lim) {
            const long long co = coff_of(c);
#pragma unroll
            for (int it = 0; it < 2; ++it) {
              const int rr = it * 16 + (lane >> 1);
              if (roff2[it] >= 0) {
                uint4 o = ld_shared_v4(stg + rr * 32 + ((cc2 ^ ((rr >> 2) & 1)) << 4));
                if (has_res) o = hadd2x4(o, ra[it]);
                *reinterpret_cast<uint4*>(p.out + roff2[it] + co) = o;
              }
            }
          }
          __syncwarp();
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(as));
        continue;
      }
      if (!LEAN) {
        mbar_wait(tfull_bar(as), aph);
        tc_fence_after();
      }
      if (p.splits > 1) {
        // split-K: raw fp32 partials -> workspace; bias/activation/residual happen in splitk_finish_kernel
        float* wrow = p.ws + ((long long)split * m_tiles * BM + (long long)m_tile * BM + row) * p.N;
        for (int ch = ch_begin; ch < ch_end; ++ch) {
          const int c0 = ch * 16;
          if (col_base + c0 >= n_out) break;
          uint32_t r[16];
          tmem_ld16(taddr + c0, r);
          tmem_ld_wait();
#pragma unroll
          for (int v4 = 0; v4 < 4; ++v4) {
            const int col = col_base + c0 + v4 * 4;
            if (col < n_out)
              *reinterpret_cast<uint4*>(wrow + col) = make_uint4(r[v4 * 4], r[v4 * 4 + 1], r[v4 * 4 + 2], r[v4 * 4 + 3]);
          }
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(as));
        continue;
      }
      if (p.vec_ok && plain_cols) {
        // ---------------- fast path: contiguous channel-last output, 16-byte stores.
        // (ncu on the first version: 243 SASS instructions per 16 columns, ~50 of them useful; small-K
        //  GEMMs were bound by this loop, not by the MMA.)  Everything tile-invariant is hoisted, loads are
        //  only issued for operands that exist, and the GEGLU gate works on packed halves.
        __half* outp = p.out + row_off;
        const __half* resp = p.residual ? p.residual + row_off : nullptr;
        const bool has_bias = p.bias != nullptr;
        const float alpha = p.alpha;
        const int act = p.act;
        for (int ch = ch_begin; ch < ch_end; ++ch) {
          const int c0 = ch * 16;
          const int col = col_base + c0;
          if (col >= n_out) break;                      // warp-uniform
          const bool two = (col + 8 < n_out);           // second 8-column half inside N (warp-uniform)
          uint32_t r[16];
          uint32_t g[16];
          tmem_ld16(taddr + c0, r);
          if (geglu) tmem_ld16(taddr + CB / 2 + c0, g);
          uint4 bu0, bu1, gu0, gu1, ra0, ra1, rs0, rs1;
          if (has_bias) {
            const __half* bp = geglu ? p.bias + (long long)n_tile * CB + c0 : p.bias + col;
            bu0 = __ldg(reinterpret_cast<const uint4*>(bp));
            if (two) bu1 = __ldg(reinterpret_cast<const uint4*>(bp + 8));
            if (geglu) {
              gu0 = __ldg(reinterpret_cast<const uint4*>(bp + CB / 2));
              if (two) gu1 = __ldg(reinterpret_cast<const uint4*>(bp + CB / 2 + 8));
            }
          }
          if (valid) {
            if (rowadd_row) {
              ra0 = __ldg(reinterpret_cast<const uint4*>(rowadd_row + col));
              if (two) ra1 = __ldg(reinterpret_cast<const uint4*>(rowadd_row + col + 8));
            }
            if (resp) {
              rs0 = __ldg(reinterpret_cast<const uint4*>(resp + col));
              if (two) rs1 = __ldg(reinterpret_cast<const uint4*>(resp + col + 8));
            }
          }
          tmem_ld_wait();
          if (valid) {
#pragma unroll
            for (int h8 = 0; h8 < 2; ++h8) {
              if (h8 == 1 && !two) break;
              float v[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[h8 * 8 + i]) * alpha;
              if (has_bias) {
                float bv[8];
                unpack8h(h8 ? bu1 : bu0, bv);
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] += bv[i];
              }
              uint4 o;
              __half2* oh = reinterpret_cast<__half2*>(&o);
              if (geglu) {
                float gt[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) gt[i] = __uint_as_float(g[h8 * 8 + i]) * alpha;
                if (has_bias) {
                  float bg[8];
                  unpack8h(h8 ? gu1 : gu0, bg);
#pragma unroll
                  for (int i = 0; i < 8; ++i) gt[i] += bg[i];
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                  // reference: x, gate = proj(x).chunk(2) are fp16 tensors; x * gelu(gate) (attention.py:50-51)
                  const __half2 a2 = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
                  const __half2 b2 = __floats2half2_rn(gt[2 * i], gt[2 * i + 1]);
                  const float2 bf = __half22float2(b2);
                  const float g0 = 0.5f * bf.x * (1.f + fast_erf(bf.x * 0.70710678118654752f));
                  const float g1 = 0.5f * bf.y * (1.f + fast_erf(bf.y * 0.70710678118654752f));
                  oh[i] = __hmul2(a2, __floats2half2_rn(g0, g1));
                }
              } else {
                if (rowadd_row) {
                  float rv[8];
                  unpack8h(h8 ? ra1 : ra0, rv);
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] += rv[i];
                }
                if (act != PFD_ACT_NONE) {
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] = act_apply(v[i], act);
                }
                if (resp) {
                  float rv[8];
                  unpack8h(h8 ? rs1 : rs0, rv);
#pragma unroll
                  for (int i = 0; i < 8; ++i) v[i] += rv[i];
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) oh[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
              }
              *reinterpret_cast<uint4*>(outp + col + h8 * 8) = o;
            }
          }
        }
        tc_fence_before();
        mbar_arrive(tempty_bar(as));
        continue;
      }
      for (int ch = ch_begin; ch < ch_end; ++ch) {
        const int c0 = ch * 16;
        if (col_base + c0 >= n_out) break;  // warp-uniform
        uint32_t r[16];
        uint32_t g[16];
        tmem_ld16(taddr + c0, r);
        if (geglu) tmem_ld16(taddr + CB / 2 + c0, g);
        // issue every global load of this chunk before waiting for TMEM
        uint4 bias_u[2], gate_u[2], radd_u[2], res_u[2];
        long long coff[2];
        bool live[2];
#pragma unroll
        for (int h8 = 0; h8 < 2; ++h8) {
          const int col = col_base + c0 + h8 * 8;
          live[h8] = valid && (col < n_out);
          if (plain_cols) {
            coff[h8] = (long long)col * p.so_c0;
          } else {
            coff[h8] = (long long)hcol * p.so_c1 + (long long)ecol * p.so_c0;
            ecol += 8;
            if (ecol >= p.cdiv) {
              ecol -= p.cdiv;
              ++hcol;
            }
          }
          bias_u[h8] = gate_u[h8] = radd_u[h8] = res_u[h8] = make_uint4(0, 0, 0, 0);
          if (col < n_out) {
            if (p.bias) {
              if (geglu) {
                bias_u[h8] = __ldg(reinterpret_cast<const uint4*>(p.bias + (long long)n_tile * CB + c0 + h8 * 8));
                gate_u[h8] = __ldg(reinterpret_cast<const uint4*>(p.bias + (long long)n_tile * CB + CB / 2 + c0 + h8 * 8));
              } else {
                bias_u[h8] = __ldg(reinterpret_cast<const uint4*>(p.bias + col));
              }
            }
            if (live[h8]) {
              if (rowadd_row) radd_u[h8] = __ldg(reinterpret_cast<const uint4*>(rowadd_row + col));
              if (p.residual && p.vec_ok) res_u[h8] = __ldg(reinterpret_cast<const uint4*>(p.residual + row_off + coff[h8]));
            }
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int h8 = 0; h8 < 2; ++h8) {
          if (!live[h8]) continue;
          const int col = col_base + c0 + h8 * 8;
          float v[8], bv[8];
          unpack8h(bias_u[h8], bv);
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] = fmaf(__uint_as_float(r[h8 * 8 + i]), p.alpha, bv[i]);
          if (geglu) {
            float gt[8], bg[8];
            unpack8h(gate_u[h8], bg);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              gt[i] = fmaf(__uint_as_float(g[h8 * 8 + i]), p.alpha, bg[i]);
              // reference rounds proj output to fp16 before the gate product (attention.py:50-51)
              const float a = __half2float(__float2half_rn(v[i]));
              const float b = __half2float(__float2half_rn(gt[i]));
              const float ge = 0.5f * b * (1.f + fast_erf(b * 0.70710678118654752f));
              v[i] = a * __half2float(__float2half_rn(ge));
            }
          } else {
            if (rowadd_row) {
              float rv[8];
              unpack8h(radd_u[h8], rv);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] += rv[i];
            }
            if (p.act != PFD_ACT_NONE) {
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] = act_apply(v[i], p.act);
            }
          }
          if (p.vec_ok) {
            if (p.residual) {
              float rv[8];
              unpack8h(res_u[h8], rv);
#pragma unroll
              for (int i = 0; i < 8; ++i) v[i] += rv[i];
            }
            uint4 o;
            __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
            for (int i = 0; i < 4; ++i) oh[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
            *reinterpret_cast<uint4*>(p.out + row_off + coff[h8]) = o;
          } else {
            // element-strided output (e.g. transposed V^T): 8 scalar stores
            const long long estep = p.so_c0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              // columns of one 8-group never straddle a head boundary (cdiv % 8 == 0 is required)
              const long long off = row_off + coff[h8] + (long long)i * estep;
              float t = v[i];
              if (p.residual) t += __half2float(p.residual[off]);
              p.out[off] = __float2half_rn(t);
            }
          }
          (void)col;
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(as));
    }
  }

  if (TMAE && warp >= 2 && lane == 0) bulk_wait_all();       // this thread's TMA stores have been performed
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------ CTA-pair kernel
// Same contraction on a PAIR of CTAs (cluster of two, tcgen05 cta_group::2): D[256 x BN] per pair, each CTA holding
// its own 128 rows of A and HALF of the B tile (BN/2 weight rows) per K block -> per-SM operand ingest drops from
// (128 + BN) x 128 B to (128 + BN/2) x 128 B per K block (BN = 256: 7.8 instead of 14 B per kFLOP), which is what the
// 3x3 convs are bound by (r1/r2 ncu: 1.5 GB of L2->SM reads per launch at 10 TB/s with the tensor pipe 65-78 % busy).
// Protocol (both CTAs run every role, identical shared-memory layouts):
//   producer  (warp 0, each CTA): waits its OWN empty barrier, loads its A tile and its B half with the cta_group::2
//             form of cp.async.bulk.tensor, whose bytes complete on the LEADER's full barrier; the leader's producer
//             arms that barrier with the bytes of both CTAs;
//   MMA       (warp 1 of the leader = cluster rank 0 only): tcgen05.mma.cta_group::2 (M = 256), tcgen05.commit with
//             cluster multicast releases the stage in both CTAs and publishes the accumulator to both epilogues;
//   epilogue  (warps 2..9, each CTA): TMA-store epilogue on the CTA's own 128 x BN accumulator in its own TMEM; one lane
//             per warp arrives on the LEADER's tmem_empty barrier (16 arrivals per tile).
// Only the TMA-store epilogue exists here (plain channel-last outputs, no GEGLU / split-K / batched B).
template <int BN>
struct GemmCfg2 {
  static constexpr int STAGE_B_BYTES = (BN / 2) * BK * 2;
  static constexpr int STAGE_BYTES = STAGE_A_BYTES + STAGE_B_BYTES;
  static constexpr int WARP_STG = epi_stg_bytes(BN, true);
  static constexpr int FIXED = 1024 + 1024 + EPI_WARPS * WARP_STG + 2 * BN * 4;
  static constexpr int RAW_STAGES = (SMEM_BUDGET - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = RAW_STAGES > 8 ? 8 : RAW_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + FIXED;
  static constexpr uint32_t TMEM_COLS = (2 * BN <= 128) ? 128u : (2 * BN <= 256 ? 256u : 512u);
  static_assert(STAGE_B_BYTES % 1024 == 0, "B half stage must keep 1024-B swizzle alignment");
  static_assert(BN % 16 == 0 && BN >= 32 && BN <= 256, "UMMA N constraint for M = 256");
  static_assert(STAGES >= 3, "too few pipeline stages");
};

template <int BN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg2<BN>;
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t base = (raw_addr + 1023u) & ~1023u;
  uint8_t* gbase = smem_raw + (base - raw_addr);
  const uint32_t smemA = base;
  const uint32_t smemB = base + STAGES * STAGE_A_BYTES;
  const uint32_t bars = base + STAGES * Cfg::STAGE_BYTES;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (STAGES + s); };
  auto tfull_bar = [&](int a) { return bars + 8u * (2 * STAGES + a); };
  auto tempty_bar = [&](int a) { return bars + 8u * (2 * STAGES + 2 + a); };
  const uint32_t tmem_slot = bars + 8u * (2 * STAGES + 4);
  auto res_bar = [&](int w) { return bars + 8u * (2 * STAGES + 5 + w); };
  volatile uint32_t* tmem_slot_g =
      reinterpret_cast<volatile uint32_t*>(gbase + STAGES * Cfg::STAGE_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < p.nseg; ++s) tma_prefetch_desc(&p.tmA[s]);
    tma_prefetch_desc(&p.tmB);
    tma_prefetch_desc(&p.tmO32);
    tma_prefetch_desc(&p.tmO16);
    if (p.residual) {
      tma_prefetch_desc(&p.tmR32);
      tma_prefetch_desc(&p.tmR16);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), 2 * EPI_WARPS);       // one lane per epilogue warp of both CTAs
    }
    for (int w = 0; w < EPI_WARPS; ++w) mbar_init(res_bar(w), 1);
    mbar_fence_init();
  }
  if (warp == 2) tmem_alloc_pair<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  cluster_sync_all();            // barriers of BOTH CTAs are initialised before any remote arrive / TMA completion
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_g;
  pdl_wait();
  pdl_launch_dependents();

  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_nb;
  const int m_pairs = (m_tiles + 1) >> 1;
  const int total_work = m_pairs * p.n_tiles;
  const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int work = cluster_id; work < total_work; work += n_clusters) {
        const int n_tile = work % p.n_tiles;
        const int m_tile = 2 * (work / p.n_tiles) + (int)rank;     // may be == m_tiles (odd tail): fully out of raster
        const int tx = m_tile % p.tiles_w;
        const int ty = (m_tile / p.tiles_w) % p.tiles_h;
        const int tn = m_tile / (p.tiles_w * p.tiles_h);
        const int x0 = tx * p.bw * p.stride;
        const int y0 = ty * p.bh * p.stride;
        const int n0 = tn * p.bn;
        int kofs = 0;
        for (int s = 0; s < p.nseg; ++s) {
          const int ntap = p.taps[s];
          for (int t = 0; t < ntap; ++t) {
            const int dy = (ntap == 9) ? (t / 3 - 1 + p.tap_off) : 0;
            const int dx = (ntap == 9) ? (t % 3 - 1 + p.tap_off) : 0;
            for (int j = 0; j < p.chunks[s]; ++j) {
              mbar_wait(empty_bar(stage), phase ^ 1u);
              if (rank == 0) mbar_expect_tx(full_bar(stage), 2 * Cfg::STAGE_BYTES);
              tma_load_4d_pair(smemA + stage * STAGE_A_BYTES, &p.tmA[s], full_bar(stage), j * BK, x0 + dx, y0 + dy, n0);
              tma_load_3d_pair(smemB + stage * Cfg::STAGE_B_BYTES, &p.tmB, full_bar(stage), kofs + j * BK,
                               n_tile * BN + (int)rank * (BN / 2), 0);
              if (++stage == STAGES) {
                stage = 0;
                phase ^= 1u;
              }
            }
            kofs += p.a_c[s];
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (one thread of the leader CTA)
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc = make_idesc_f16_pair(BN);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int work = cluster_id; work < total_work; work += n_clusters, ++it) {
        const int as = it & 1;
        const uint32_t aph = (it >> 1) & 1;
        mbar_wait(tempty_bar(as), aph ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * BN;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint64_t adesc = make_sw128_kmajor_desc(smemA + stage * STAGE_A_BYTES);
          const uint64_t bdesc = make_sw128_kmajor_desc(smemB + stage * Cfg::STAGE_B_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_f16_pair(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit_pair(empty_bar(stage));
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit_pair(tfull_bar(as));
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue (warps 2..9 of both CTAs)
    const int q = warp & 3;
    const int half_id = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const int rdx = row % p.bw;
    const int rdy = (row / p.bw) % p.bh;
    const int rdn = row / (p.bw * p.bh);
    constexpr int nch = BN / 16;
    const int ch_begin = half_id == 0 ? 0 : (nch + 1) / 2;
    const int ch_end = half_id == 0 ? (nch + 1) / 2 : nch;
    const int cbeg = ch_begin * 16, cend = ch_end * 16;
    const uint32_t fixed0 = base + STAGES * Cfg::STAGE_BYTES + 1024;
    uint32_t res_phase = 0;
    int it = 0;
    for (int work = cluster_id; work < total_work; work += n_clusters, ++it) {
      const int as = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      const int n_tile = work % p.n_tiles;
      const int m_tile = 2 * (work / p.n_tiles) + (int)rank;
      EpiTile e;
      e.q = q; e.lane = lane;
      e.tx = m_tile % p.tiles_w;
      e.ty = (m_tile / p.tiles_w) % p.tiles_h;
      e.tn = m_tile / (p.tiles_w * p.tiles_h);
      const int x = e.tx * p.bw + rdx, y = e.ty * p.bh + rdy, n = e.tn * p.bn + rdn;
      e.valid = (x < p.W) && (y < p.H) && (n < p.NB);
      e.cbeg = cbeg; e.n32 = (cend - cbeg) >> 5; e.tail16 = ((cend - cbeg) & 16) != 0;
      e.col_base = n_tile * BN; e.n_lim = p.N;
      e.has_res = p.residual != nullptr;
      e.stg = fixed0 + (warp - 2) * Cfg::WARP_STG;
      e.rbar = res_bar(warp - 2);
      e.tfull = tfull_bar(as);
      e.aph = aph;
      e.taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + as * BN;
      e.sbias = fixed0 + EPI_WARPS * Cfg::WARP_STG + as * (BN * 4);
      e.alpha = p.alpha; e.act = p.act;
      e.rowadd_row = (p.rowadd && e.valid) ? p.rowadd + (long long)n * p.rowadd_ld : nullptr;
      e.sk_mode = 0; e.sk_slot = 0; e.sk_t = 0; e.sk_kb0 = 0; e.stg_warp = warp - 2;
      const int et = threadIdx.x - 64;
      if (et < BN) {
        const int c = e.col_base + et;
        const float b = (p.bias != nullptr && c < p.N) ? __half2float(__ldg(p.bias + c)) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(e.sbias + et * 4), "f"(b) : "memory");
      }
      tma_store_epilogue<BN, false>(p, e, res_phase);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(tempty_bar(as));
    }
    if (lane == 0) bulk_wait_all();
  }

  tc_fence_before();
  cluster_sync_all();            // neither CTA may leave (or free TMEM) while the pair's MMAs / remote arrives are in flight
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_pair<Cfg::TMEM_COLS>(tmem_base);
  }
}

// Split-K second pass: sum the fp32 partials of all splits and apply the fused epilogue
// (bias, per-image row add, activation, residual) with the same generic output addressing.
__global__ void __launch_bounds__(256)
splitk_finish_kernel(const __grid_constant__ GemmParams p) {
  pdl_wait();
  pdl_launch_dependents();
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_nb;
  const long long rows_pad = (long long)m_tiles * BM;
  const int vecs = p.N / 8;
  const long long total = rows_pad * vecs;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % vecs);
    const long long prow = i / vecs;
    const int m_tile = (int)(prow / BM), row = (int)(prow % BM);
    const int tx = m_tile % p.tiles_w;
    const int ty = (m_tile / p.tiles_w) % p.tiles_h;
    const int tn = m_tile / (p.tiles_w * p.tiles_h);
    const int x = tx * p.bw + row % p.bw;
    const int y = ty * p.bh + (row / p.bw) % p.bh;
    const int n = tn * p.bn + row / (p.bw * p.bh);
    if (x >= p.W || y >= p.H || n >= p.NB) continue;
    const int col = v * 8;
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.f;
    for (int s = 0; s < p.splits; ++s) {
      const float4* src = reinterpret_cast<const float4*>(p.ws + ((long long)s * rows_pad + prow) * p.N + col);
      const float4 a = __ldg(src), b = __ldg(src + 1);
      acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
      acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
    }
    float bv[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) bv[k] = 0.f;
    if (p.bias) load8h(p.bias + col, bv);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = fmaf(acc[k], p.alpha, bv[k]);
    if (p.rowadd) {
      float rv[8];
      load8h(p.rowadd + (long long)n * p.rowadd_ld + col, rv);
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] += rv[k];
    }
    if (p.act != PFD_ACT_NONE) {
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = act_apply(acc[k], p.act);
    }
    const long long row_off = (long long)(n / p.ndiv) * p.so_n1 + (long long)(n % p.ndiv) * p.so_n0 +
                              (long long)y * p.so_y + (long long)x * p.so_x;
    const long long coff = (long long)(col / p.cdiv) * p.so_c1 + (long long)(col % p.cdiv) * p.so_c0;
    if (p.vec_ok) {
      if (p.residual) {
        float rv[8];
        load8h(p.residual + row_off + coff, rv);
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] += rv[k];
      }
      uint4 o;
      __half2* oh = reinterpret_cast<__half2*>(&o);
#pragma unroll
      for (int k = 0; k < 4; ++k) oh[k] = __floats2half2_rn(acc[2 * k], acc[2 * k + 1]);
      *reinterpret_cast<uint4*>(p.out + row_off + coff) = o;
    } else {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const long long off = row_off + coff + (long long)k * p.so_c0;
        float t = acc[k];
        if (p.residual) t += __half2float(p.residual[off]);
        p.out[off] = __float2half_rn(t);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ host
constexpr size_t SPLITK_WS_BYTES = 64ull << 20;
constexpr size_t SK_FLAG_BYTES = 4096;          // stream-K flags live at the end of the workspace
// One fp32 split-K workspace per DEVICE, allocated by the first pfd_gemm_f16 call on that device that is not
// inside a stream capture (cudaMalloc is illegal while capturing) - i.e. in the eager warm-up pass that every
// graph-captured path of this package runs first - and then shared by the eager and the captured launches, so
// that graph replay and eager execution choose the same split configuration (r1 advisor finding: the old
// per-stream map was always empty on torch's capture stream, silently disabling split-K in every replayed path).
// Launches of one device are stream-ordered by the callers (one request at a time, SURVEY.md 8b), so one buffer
// per device is enough.
static float* splitk_workspace(cudaStream_t st) {
  constexpr int MAX_DEV = 64;
  static std::mutex mu;
  static float* ws[MAX_DEV] = {nullptr};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= MAX_DEV) return nullptr;
  std::lock_guard<std::mutex> lk(mu);
  if (ws[dev]) return ws[dev];
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess || cs != cudaStreamCaptureStatusNone) {
    (void)cudaGetLastError();
    return nullptr;
  }
  float* pnew = nullptr;
  if (cudaMalloc(&pnew, SPLITK_WS_BYTES) != cudaSuccess) {
    (void)cudaGetLastError();
    return nullptr;
  }
  // the last SK_FLAG_BYTES hold the stream-K ready flags: zero once, every consumer resets the flags it has read
  if (cudaMemset(reinterpret_cast<char*>(pnew) + SPLITK_WS_BYTES - SK_FLAG_BYTES, 0, SK_FLAG_BYTES) != cudaSuccess ||
      cudaDeviceSynchronize() != cudaSuccess) {
    (void)cudaGetLastError();
    cudaFree(pnew);
    return nullptr;
  }
  ws[dev] = pnew;
  return pnew;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = reinterpret_cast<EncodeTiledFn>(p);
    }
  }
  return fn;
}

static int encode_map(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims,
                      const cuuint64_t* strides_bytes, const cuuint32_t* box,
                      const cuuint32_t* estr, const char* what,
                      CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, const_cast<void*>(ptr), dims,
                  strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    return set_error(
        "tensor map (%s) encode failed: CUresult %d rank %d dims[%llu,%llu,%llu,%llu] "
        "strides[%llu,%llu,%llu] box[%u,%u,%u,%u] ptr %p",
        what, (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
        (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
        (unsigned long long)strides_bytes[0], (unsigned long long)(rank > 2 ? strides_bytes[1] : 0),
        (unsigned long long)(rank > 3 ? strides_bytes[2] : 0), box[0], box[1], rank > 2 ? box[2] : 0,
        rank > 3 ? box[3] : 0, ptr);
  }
  return 0;
}

static inline long long cdivll(long long a, long long b) { return (a + b - 1) / b; }

template <int BN, bool LEAN, bool TMAE, bool SK = false>
static int launch_gemm_t(const GemmParams& p, int grid, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, TMAE>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<BN, LEAN, TMAE, SK>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return set_error("cudaFuncSetAttribute(gemm BN=%d): %s", BN, cudaGetErrorString(e));
    attr_done = true;
  }
  launch_k(gemm_tc_kernel<BN, LEAN, TMAE, SK>, dim3(grid), dim3(GEMM_THREADS), Cfg::SMEM_BYTES, stream, p);
  return check_launch("pfd_gemm_f16");
}

// Output (and residual) rasters as TMA tensor maps for the TMA-store epilogue: dims {N, W, H, NB}, one box = the 32
// consecutive tile rows of an epilogue warp (sbw x sbh x sbn pixels) x 32 or 16 channels.
static int encode_epilogue_maps(GemmParams& p, const pfd_gemm_desc* d) {
  const int sbw = p.bw < 32 ? p.bw : 32;
  const int sbh = p.bh < 32 / sbw ? p.bh : 32 / sbw;
  const int sbn = 32 / (sbw * sbh);
  const long long sx = d->so_x, sy = d->H > 1 ? d->so_y : sx * d->W, sn = d->NB > 1 ? d->so_n1 : sy * d->H;
  cuuint64_t dims[4] = {(cuuint64_t)d->N, (cuuint64_t)d->W, (cuuint64_t)d->H, (cuuint64_t)d->NB};
  cuuint64_t strides[3] = {(cuuint64_t)sx * 2, (cuuint64_t)sy * 2, (cuuint64_t)sn * 2};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  cuuint32_t box32[4] = {32, (cuuint32_t)sbw, (cuuint32_t)sbh, (cuuint32_t)sbn};
  cuuint32_t box16[4] = {16, (cuuint32_t)sbw, (cuuint32_t)sbh, (cuuint32_t)sbn};
  if (int rc = encode_map(&p.tmO32, d->out, 4, dims, strides, box32, estr, "out32", CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  if (int rc = encode_map(&p.tmO16, d->out, 4, dims, strides, box16, estr, "out16", CU_TENSOR_MAP_SWIZZLE_32B)) return rc;
  if (d->residual) {
    if (int rc = encode_map(&p.tmR32, d->residual, 4, dims, strides, box32, estr, "res32", CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
    if (int rc = encode_map(&p.tmR16, d->residual, 4, dims, strides, box16, estr, "res16", CU_TENSOR_MAP_SWIZZLE_32B)) return rc;
  }
  return 0;
}

static inline bool gemm_lean_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("PFD_NO_LEAN_EPI");
    v = (e && e[0] == '1') ? 0 : 1;
  }
  return v == 1;
}

template <int BN>
static int launch_gemm(GemmParams& p, int grid, cudaStream_t stream, const pfd_gemm_desc* d) {
  const bool lean = gemm_lean_enabled() && p.vec_ok && p.splits == 1;
  // TMA-store epilogue: plain channel-last output raster (no head / batch split), not GEGLU, tile staging fits (BN <= 192)
  bool tmae = false;
  if constexpr (BN <= 192) {
    tmae = lean && p.cdiv >= p.N && p.ndiv == 1 && p.act != PFD_ACT_GEGLU && option("gemm_tma_epi", 1) &&
           (d->H == 1 || d->so_y >= (long long)d->so_x * d->W) && (d->NB == 1 || d->so_n1 > 0);
    if (tmae && encode_epilogue_maps(p, d)) {
      tmae = false;                       // raster not expressible as a tensor map: keep the register epilogue
      g_last_error.clear();
    }
    // stream-K tail (see gemm_work), OPT-IN (gemm_streamk = 1): the tiles of the last, partially filled wave are spread
    // over all SMs by K range; every tile of the tail must be covered by at most 6 contributors.  Correct and
    // deterministic, but measured 0.84-0.99x on the UNet's convs / long-K Linears (profiles/r2_ab_gemm_streamk.log): the
    // per-CTA cost of the hand-off (contributor epilogue + release visibility + gather + two extra pipeline fills,
    // ~10 us) is as large as the 0.14-0.54 tile it saves at these tile times (13-45 us).
    p.sk_R = 0;
    p.sk_dp_tiles = 0;
    if (tmae && option("gemm_streamk", 0)) {
      const int G = num_sms();
      const long long T = (long long)p.tiles_w * p.tiles_h * p.tiles_nb * p.n_tiles;
      const long long R = T % G, waves = (T + G - 1) / G;
      float* ws = splitk_workspace(stream);
      const size_t need = (size_t)2 * G * BM * BN * sizeof(float);
      if (ws && R > 0 && p.num_kb >= 16 && R * 6 >= G && (size_t)2 * G * sizeof(int) <= SK_FLAG_BYTES &&
          need <= SPLITK_WS_BYTES - SK_FLAG_BYTES && (double)T / G < 0.95 * (double)waves) {
        p.sk_dp_tiles = (int)(T - R);
        p.sk_R = (int)R;
        p.sk_ws = ws;
        p.sk_flags = reinterpret_cast<int*>(reinterpret_cast<char*>(ws) + SPLITK_WS_BYTES - SK_FLAG_BYTES);
        grid = G;
      }
    }
  }
  static int trace = -1;
  if (trace < 0) {
    const char* e = getenv("PFD_GEMM_TRACE");
    trace = (e && e[0] == '1') ? 1 : 0;
  }
  if (trace)   // one line per launch, joined with an ncu launch list by tools/gemm_breakdown.py
    fprintf(stderr, "GEMMTRACE M=%lld N=%d K=%d nseg=%d taps=%d stride=%d act=%d bias=%d res=%d rowadd=%d BN=%d lean=%d "
            "splits=%d grid=%d batched=%d vec=%d plain=%d tmae=%d sk=%d\n", (long long)p.W * p.H * p.NB, p.N, p.num_kb * BK, p.nseg,
            p.taps[0], p.stride, p.act, p.bias != nullptr, p.residual != nullptr, p.rowadd != nullptr, BN, (int)lean,
            p.splits, grid, p.b_batched, p.vec_ok, (int)(p.cdiv >= p.N), (int)tmae, p.sk_R);
  if constexpr (BN <= 192) {
    if (tmae && p.sk_R > 0) return launch_gemm_t<BN, true, true, true>(p, grid, stream);
    if (tmae) return launch_gemm_t<BN, true, true>(p, grid, stream);
  }
  return lean ? launch_gemm_t<BN, true, false>(p, grid, stream) : launch_gemm_t<BN, false, false>(p, grid, stream);
}

template <int BN>
static int launch_gemm_pair(GemmParams& p, int clusters, cudaStream_t stream, const pfd_gemm_desc* d) {
  using Cfg = GemmCfg2<BN>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc2_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return set_error("cudaFuncSetAttribute(gemm pair BN=%d): %s", BN, cudaGetErrorString(e));
    attr_done = true;
  }
  if (int rc = encode_epilogue_maps(p, d)) return rc;
  static int trace = -1;
  if (trace < 0) {
    const char* e = getenv("PFD_GEMM_TRACE");
    trace = (e && e[0] == '1') ? 1 : 0;
  }
  if (trace)
    fprintf(stderr, "GEMMTRACE M=%lld N=%d K=%d nseg=%d taps=%d stride=%d act=%d bias=%d res=%d rowadd=%d BN=%d lean=P "
            "splits=1 grid=%d batched=0 vec=1 plain=1 tmae=2\n", (long long)p.W * p.H * p.NB, p.N, p.num_kb * BK, p.nseg,
            p.taps[0], p.stride, p.act, p.bias != nullptr, p.residual != nullptr, p.rowadd != nullptr, BN, 2 * clusters);
  launch_k(gemm_tc2_kernel<BN>, dim3(2 * clusters), dim3(GEMM_THREADS), Cfg::SMEM_BYTES, stream, p);
  return check_launch("pfd_gemm_f16(pair)");
}

}  // namespace pfd

using namespace pfd;

extern "C" PFD_API int pfd_gemm_f16(const pfd_gemm_desc* d) {
  if (!d) return set_error("pfd_gemm_f16: null descriptor");
  if (d->nseg < 1 || d->nseg > PFD_MAX_SEG) return set_error("pfd_gemm_f16: nseg %d out of range", d->nseg);
  if (d->N <= 0 || d->N % 8) return set_error("pfd_gemm_f16: N=%d must be a positive multiple of 8", d->N);
  if (d->K % 8) return set_error("pfd_gemm_f16: K pitch %lld must be a multiple of 8", (long long)d->K);
  if (d->W <= 0 || d->H <= 0 || d->NB <= 0) return set_error("pfd_gemm_f16: empty output raster");
  if (d->stride != 1 && d->stride != 2) return set_error("pfd_gemm_f16: stride %d unsupported", d->stride);
  if (d->tap_off != 0 && d->tap_off != 1) return set_error("pfd_gemm_f16: tap_off %d unsupported", d->tap_off);
  if (!d->out || !d->b_ptr) return set_error("pfd_gemm_f16: null out/b pointer");
  long long ktot = 0;
  for (int s = 0; s < d->nseg; ++s) {
    if (d->taps[s] != 1 && d->taps[s] != 9) return set_error("pfd_gemm_f16: taps[%d]=%d", s, d->taps[s]);
    if (d->a_c[s] <= 0 || d->a_c[s] % 8) return set_error("pfd_gemm_f16: a_c[%d]=%d must be a multiple of 8", s, d->a_c[s]);
    if (!d->a_ptr[s]) return set_error("pfd_gemm_f16: a_ptr[%d] is null", s);
    if ((reinterpret_cast<uintptr_t>(d->a_ptr[s]) & 15) || (d->a_sx[s] % 8) || (d->a_sy[s] % 8) || (d->a_sn[s] % 8))
      return set_error("pfd_gemm_f16: A segment %d not 16-byte aligned/strided", s);
    ktot += (long long)d->taps[s] * d->a_c[s];
  }
  if (ktot > d->K) return set_error("pfd_gemm_f16: segments cover K=%lld > pitch %lld", ktot, (long long)d->K);
  if (reinterpret_cast<uintptr_t>(d->b_ptr) & 15) return set_error("pfd_gemm_f16: B not 16-byte aligned");
  const bool geglu = d->act == PFD_ACT_GEGLU;

  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.nseg = d->nseg;
  p.stride = d->stride;
  p.tap_off = d->tap_off;
  p.W = d->W; p.H = d->H; p.NB = d->NB; p.N = d->N;
  p.b_batched = d->b_batch_stride != 0;
  p.alpha = d->alpha;
  p.act = d->act;
  p.bias = static_cast<const __half*>(d->bias);
  p.rowadd = static_cast<const __half*>(d->rowadd);
  p.residual = static_cast<const __half*>(d->residual);
  p.rowadd_ld = d->rowadd_ld > 0 ? d->rowadd_ld : d->N;
  p.out = static_cast<__half*>(d->out);
  p.so_n1 = d->so_n1; p.so_n0 = d->so_n0; p.so_y = d->so_y; p.so_x = d->so_x;
  p.so_c1 = d->so_c1; p.so_c0 = d->so_c0;
  p.ndiv = d->ndiv > 0 ? d->ndiv : 1;
  p.cdiv = d->cdiv > 0 ? d->cdiv : (1 << 30);
  p.vec_ok = (d->so_c0 == 1) && (p.cdiv % 8 == 0) && (d->so_n1 % 8 == 0) && (d->so_n0 % 8 == 0) &&
             (d->so_y % 8 == 0) && (d->so_x % 8 == 0) && (d->so_c1 % 8 == 0) &&
             ((reinterpret_cast<uintptr_t>(d->out) & 15) == 0) &&
             ((reinterpret_cast<uintptr_t>(d->residual) & 15) == 0);
  if ((reinterpret_cast<uintptr_t>(d->bias) & 15) || (reinterpret_cast<uintptr_t>(d->rowadd) & 15) || (d->rowadd_ld % 8))
    return set_error("pfd_gemm_f16: bias/rowadd must be 16-byte aligned");

  // ---- output raster tiling: 128 rows = bw x bh x bn pixels, minimise padded work
  int bw = 128, bh = 1, bn = 1;
  if (!p.b_batched) {
    long long best = -1;
    for (int cw = 128; cw >= 1; cw >>= 1) {
      if (cw * d->stride > 256) continue;
      for (int ch = 128 / cw; ch >= 1; ch >>= 1) {
        if (ch * d->stride > 256) continue;
        int cn = 128 / (cw * ch);
        long long cost = cdivll(d->W, cw) * cdivll(d->H, ch) * cdivll(d->NB, cn);
        if (best < 0 || cost < best) {
          best = cost; bw = cw; bh = ch; bn = cn;
        }
      }
    }
  }
  p.bw = bw; p.bh = bh; p.bn = bn;
  p.tiles_w = (int)cdivll(d->W, bw);
  p.tiles_h = (int)cdivll(d->H, bh);
  p.tiles_nb = (int)cdivll(d->NB, bn);
  const long long m_tiles = (long long)p.tiles_w * p.tiles_h * p.tiles_nb;

  // ---- N tile: minimise (waves x per-tile cost)
  const int cands[5] = {256, 192, 160, 128, 64};
  int BNsel = 128;
  double best_cost = -1;
  const int sms = num_sms();
  for (int i = 0; i < 5; ++i) {
    const int bn_c = cands[i];
    if (geglu && (d->N % bn_c)) continue;
    if (d->bn_force && d->bn_force != bn_c) continue;
    const long long nt = cdivll(d->N, bn_c);
    const long long tiles = m_tiles * nt;
    const double waves = (double)cdivll(tiles, sms);
    const double cost = waves * (bn_c + 24);
    if (best_cost < 0 || cost < best_cost - 1e-9) {
      best_cost = cost; BNsel = bn_c;
    }
  }
  if (best_cost < 0) return set_error("pfd_gemm_f16: no valid N tile (bn_force=%d, N=%d, geglu=%d)", d->bn_force, d->N, (int)geglu);
  p.n_tiles = (int)cdivll(d->N, BNsel);
  p.splits = 1;

  // ---- CTA-pair kernel (cta_group::2, 256 x BN per pair): long-K contractions with a plain channel-last output whose
  //      operand ingest, not the epilogue, is the bound (3x3 convs, K >= 1024 Linears) and that fill the 74 pairs
  int k_blocks = 0;
  for (int s = 0; s < d->nseg; ++s) k_blocks += d->taps[s] * ((d->a_c[s] + BK - 1) / BK);
  const int pair_mode = option("gemm_pair", 0);
  bool use_pair = pair_mode > 0 && !geglu && !p.b_batched && !d->bn_force && p.vec_ok && p.cdiv >= p.N && p.ndiv == 1 &&
                  gemm_lean_enabled() && (d->H == 1 || d->so_y >= (long long)d->so_x * d->W) &&
                  (d->NB == 1 || d->so_n1 > 0) && m_tiles >= 2 && k_blocks >= (pair_mode > 1 ? 1 : 16);
  if (use_pair) {
    const long long m_pairs = (m_tiles + 1) / 2;
    const int pc[3] = {256, 160, 128};
    double pbest = -1;
    int pbn = 160;
    for (int i = 0; i < 3; ++i) {
      const long long tiles = m_pairs * cdivll(d->N, pc[i]);
      const double cost = (double)cdivll(tiles, sms / 2) * (pc[i] + 24);
      if (pbest < 0 || cost < pbest - 1e-9) {
        pbest = cost; pbn = pc[i];
      }
    }
    // the machine must be filled: at least one full wave of pairs (smaller problems keep split-K / the single-CTA tiles)
    if (m_pairs * cdivll(d->N, pbn) * 2 < sms && pair_mode < 2) use_pair = false;
    else {
      BNsel = pbn;
      p.n_tiles = (int)cdivll(d->N, BNsel);
    }
  }

  // ---- tensor maps
  int num_kb = 0;
  for (int s = 0; s < d->nseg; ++s) {
    p.taps[s] = d->taps[s];
    p.a_c[s] = d->a_c[s];
    p.chunks[s] = (d->a_c[s] + BK - 1) / BK;
    num_kb += p.taps[s] * p.chunks[s];
    cuuint64_t dims[4] = {(cuuint64_t)d->a_c[s], (cuuint64_t)d->in_w, (cuuint64_t)d->in_h, (cuuint64_t)d->NB};
    cuuint64_t strides[3] = {(cuuint64_t)d->a_sx[s] * 2, (cuuint64_t)d->a_sy[s] * 2, (cuuint64_t)d->a_sn[s] * 2};
    cuuint32_t box[4] = {(cuuint32_t)BK, (cuuint32_t)(bw * d->stride), (cuuint32_t)(bh * d->stride), (cuuint32_t)bn};
    cuuint32_t estr[4] = {1, (cuuint32_t)d->stride, (cuuint32_t)d->stride, 1};
    if (int rc = encode_map(&p.tmA[s], d->a_ptr[s], 4, dims, strides, box, estr, "A")) return rc;
  }
  p.num_kb = num_kb;
  p.kb_per_split = num_kb;
  cudaStream_t st = static_cast<cudaStream_t>(d->stream);
  float* const skws = splitk_workspace(st);     // allocated by the first eager call on this device
  // ---- split-K for long-K problems that cannot fill the machine (8x8-level convs): fewer, wider N tiles
  //      (less A re-read through L2) x several K slices, fp32 partials reduced by splitk_finish_kernel.
  if (!use_pair && !geglu && !d->bn_force && num_kb >= 32) {
    int bn_sk = 128;
    const int sk_cands[4] = {256, 192, 160, 128};
    for (int i = 0; i < 4; ++i)
      if (d->N % sk_cands[i] == 0) {
        bn_sk = sk_cands[i];
        break;
      }
    const long long nt_sk = cdivll(d->N, bn_sk);
    const long long tiles_sk = m_tiles * nt_sk;
    if (tiles_sk * 2 <= sms) {
      int splits = (int)(sms / tiles_sk);
      if (splits > 8) splits = 8;
      if (splits > num_kb / 8) splits = num_kb / 8;
      const size_t need = (size_t)splits * (size_t)m_tiles * BM * (size_t)d->N * sizeof(float);
      if (splits >= 2 && need <= SPLITK_WS_BYTES - SK_FLAG_BYTES) {
        float* ws = skws;
        if (ws) {
          BNsel = bn_sk;
          p.n_tiles = (int)nt_sk;
          p.splits = splits;
          p.kb_per_split = (num_kb + splits - 1) / splits;
          p.splits = (num_kb + p.kb_per_split - 1) / p.kb_per_split;
          p.ws = ws;
        }
      }
    }
  }
  {
    const long long nbatch = p.b_batched ? d->NB : 1;
    cuuint64_t dims[3] = {(cuuint64_t)d->K, (cuuint64_t)d->N, (cuuint64_t)nbatch};
    const long long bs = p.b_batched ? d->b_batch_stride : (long long)d->K * d->N;
    cuuint64_t strides[2] = {(cuuint64_t)d->K * 2, (cuuint64_t)bs * 2};
    cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)(use_pair ? BNsel / 2 : BNsel), 1};   // pair: each CTA loads half
    cuuint32_t estr[3] = {1, 1, 1};
    if (int rc = encode_map(&p.tmB, d->b_ptr, 3, dims, strides, box, estr, "B")) return rc;
  }
  if (use_pair) {
    const long long work = ((m_tiles + 1) / 2) * p.n_tiles;
    const int clusters = (int)(work < sms / 2 ? work : sms / 2);
    switch (BNsel) {
      case 128: return launch_gemm_pair<128>(p, clusters, st, d);
      case 160: return launch_gemm_pair<160>(p, clusters, st, d);
      default: return launch_gemm_pair<256>(p, clusters, st, d);
    }
  }

  const long long total = m_tiles * p.n_tiles * p.splits;
  int grid = (int)(total < sms ? total : sms);
  int rc;
  switch (BNsel) {
    case 64: rc = launch_gemm<64>(p, grid, st, d); break;
    case 128: rc = launch_gemm<128>(p, grid, st, d); break;
    case 160: rc = launch_gemm<160>(p, grid, st, d); break;
    case 192: rc = launch_gemm<192>(p, grid, st, d); break;
    default: rc = launch_gemm<256>(p, grid, st, d); break;
  }
  if (rc || p.splits == 1) return rc;
  const long long vec_items = m_tiles * BM * (long long)(d->N / 8);
  long long fgrid = (vec_items + 255) / 256;
  if (fgrid > 8LL * sms) fgrid = 8LL * sms;
  launch_k(splitk_finish_kernel, dim3((unsigned)fgrid), dim3(256), 0, st, p);
  return check_launch("pfd_gemm_f16(split-K finish)");
}
