// Row-wise HBM-bound kernels of the transformer block and the latent head:
//   gain-only LayerNorm fwd/bwd   (reference x_clip/x_clip.py:112-121; used at :126,:210,:193,:271-272)
//   l2-normalise fwd/bwd          (reference :54-55, called at :715,:724)
//   fp32 -> bf16 cast             (weights are kept fp32 by the module; MMA operands are bf16)
//
// One warp owns one row; a lane owns 16-byte vectors (8 bf16) strided by 32 lanes so every
// warp-wide access is a fully coalesced 512-byte segment.  Row statistics are reduced with
// warp shuffles in fp32.  Column reductions (gain gradients) are accumulated per lane in
// registers over the rows a warp visits, combined across the block in shared memory and
// added to the fp32 output with one atomic per column per block.
#include "common.cuh"
#include "host.h"

namespace xclip {

constexpr int kRowThreads = 256;
constexpr int kRowWarps = kRowThreads / 32;

__device__ __forceinline__ void load8(const bf16* p, float (&f)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z),
         d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z),
         d = unpack_bf16x2(u.w);
  f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}

__device__ __forceinline__ void store8(bf16* p, const float (&f)[8]) {
  uint4 u;
  u.x = pack_bf16x2(f[0], f[1]); u.y = pack_bf16x2(f[2], f[3]);
  u.z = pack_bf16x2(f[4], f[5]); u.w = pack_bf16x2(f[6], f[7]);
  *reinterpret_cast<uint4*>(p) = u;
}

__device__ __forceinline__ void loadf8(const float* p, float (&f)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p);
  const float4 b = *reinterpret_cast<const float4*>(p + 4);
  f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
}

__device__ __forceinline__ void storef8(float* p, const float (&f)[8]) {
  *reinterpret_cast<float4*>(p) = make_float4(f[0], f[1], f[2], f[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(f[4], f[5], f[6], f[7]);
}

__device__ __forceinline__ float bf16_round(float v) {
  return __bfloat162float(__float2bfloat16_rn(v));
}

// Adds the per-lane column partials of all warps of the block and issues one atomicAdd per column.
template <int NV>
__device__ __forceinline__ void flush_column_partials(float (&acc)[NV][8], float* dst,
                                                      float* smem /* [NV*256] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < NV * 256; i += kRowThreads) smem[i] = 0.f;
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NV; ++j)
#pragma unroll
    for (int e = 0; e < 8; ++e) atomicAdd(&smem[(j * 32 + lane) * 8 + e], acc[j][e]);
  (void)warp;
  __syncthreads();
  for (int i = threadIdx.x; i < NV * 256; i += kRowThreads) atomicAdd(dst + i, smem[i]);
}

// ---------------------------------------------------------------------------
// LayerNorm forward:  out = LN(x) * g (+ res);  optionally out2 = LN(bf16(out)) * g2
// stats = (mean, rstd) per row of the FIRST norm, stats2 of the second.
// ---------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kRowThreads)
ln_fwd_kernel(const bf16* __restrict__ x, long long ldx, const float* __restrict__ g,
              const bf16* __restrict__ res, long long ldres, bf16* __restrict__ out,
              long long ldo, float* __restrict__ stats, const float* __restrict__ g2,
              bf16* __restrict__ out2, long long ldo2, float* __restrict__ stats2, int rows,
              float eps) {
  constexpr int D = NV * 256;
  const int lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  const int warp_stride = gridDim.x * kRowWarps;
  constexpr bool kPipelined = NV <= 3;   // next row's vectors in flight while this row is reduced
  uint4 nx[NV];
  if (kPipelined && warp_global < rows) {
#pragma unroll
    for (int j = 0; j < NV; ++j)
      nx[j] = *reinterpret_cast<const uint4*>(x + warp_global * ldx + (j * 32 + lane) * 8);
  }
  for (int row = warp_global; row < rows; row += warp_stride) {
    float v[NV][8];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      if (kPipelined) unpack8(nx[j], v[j]);
      else load8(x + row * ldx + (j * 32 + lane) * 8, v[j]);
#pragma unroll
      for (int e = 0; e < 8; ++e) s += v[j][e];
    }
    if (kPipelined && row + warp_stride < rows) {
#pragma unroll
      for (int j = 0; j < NV; ++j)
        nx[j] = *reinterpret_cast<const uint4*>(x + (row + warp_stride) * ldx + (j * 32 + lane) * 8);
    }
    const float mean = warp_sum(s) * (1.f / D);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j)
#pragma unroll
      for (int e = 0; e < 8; ++e) { const float c = v[j][e] - mean; q += c * c; }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / D) + eps);
    if (lane == 0 && stats != nullptr) {
      stats[2 * (long long)row] = mean;
      stats[2 * (long long)row + 1] = rstd;
    }
    float s2 = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int col = (j * 32 + lane) * 8;
      float gg[8];
      loadf8(g + col, gg);
      float r[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (res != nullptr) load8(res + row * ldres + col, r);
#pragma unroll
      for (int e = 0; e < 8; ++e) v[j][e] = (v[j][e] - mean) * rstd * gg[e] + r[e];
      store8(out + row * ldo + col, v[j]);
      if (g2 != nullptr) {
#pragma unroll
        for (int e = 0; e < 8; ++e) { v[j][e] = bf16_round(v[j][e]); s2 += v[j][e]; }
      }
    }
    if (g2 != nullptr) {
      const float mean2 = warp_sum(s2) * (1.f / D);
      float q2 = 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j)
#pragma unroll
        for (int e = 0; e < 8; ++e) { const float c = v[j][e] - mean2; q2 += c * c; }
      const float rstd2 = rsqrtf(warp_sum(q2) * (1.f / D) + eps);
      if (lane == 0 && stats2 != nullptr) {
        stats2[2 * (long long)row] = mean2;
        stats2[2 * (long long)row + 1] = rstd2;
      }
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const int col = (j * 32 + lane) * 8;
        float gg[8];
        loadf8(g2 + col, gg);
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = (v[j][e] - mean2) * rstd2 * gg[e];
        store8(out2 + row * ldo2 + col, o);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// LayerNorm backward: dx = rstd * (g*dy - mean(g*dy) - xhat * mean(g*dy*xhat)) (+ add)
//                     dg += sum_rows dy * xhat
// ---------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kRowThreads)
ln_bwd_kernel(const bf16* __restrict__ dy, long long lddy, const bf16* __restrict__ x,
              long long ldx, const float* __restrict__ stats, const float* __restrict__ g,
              const bf16* __restrict__ add, long long ldadd, bf16* __restrict__ dx,
              long long lddx, float* __restrict__ dg, int rows) {
  constexpr int D = NV * 256;
  __shared__ float red[NV * 256];
  const int lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  const int warp_stride = gridDim.x * kRowWarps;
  float dgacc[NV][8];
#pragma unroll
  for (int j = 0; j < NV; ++j)
#pragma unroll
    for (int e = 0; e < 8; ++e) dgacc[j][e] = 0.f;
  float gg[NV][8];
#pragma unroll
  for (int j = 0; j < NV; ++j) loadf8(g + (j * 32 + lane) * 8, gg[j]);

  // software pipeline: x, dy (and the residual gradient) of the warp's NEXT row are in flight
  // while the current row is reduced
  constexpr bool kPipelined = NV <= 2;   // wider rows would spill: they load just in time
  uint4 nx[NV], nd[NV], na[NV];
  float nmean = 0.f, nrstd = 0.f;
  auto prefetch = [&](int r) {
    if (r < rows) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const int col = (j * 32 + lane) * 8;
        nx[j] = *reinterpret_cast<const uint4*>(x + r * ldx + col);
        nd[j] = *reinterpret_cast<const uint4*>(dy + r * lddy + col);
        if (kPipelined && add != nullptr)
          na[j] = *reinterpret_cast<const uint4*>(add + r * ldadd + col);
      }
      nmean = stats[2 * (long long)r];
      nrstd = stats[2 * (long long)r + 1];
    }
  };
  // wide rows (no register pipeline): pull the next row towards L2 instead - no registers held,
  // the just-in-time loads then see L2 instead of HBM latency
  auto prefetch_l2 = [&](long long r) {
    if (r < rows && (lane & 7) == 0) {
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const int col = (j * 32 + lane) * 8;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(x + r * ldx + col));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(dy + r * lddy + col));
        if (add != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(add + r * ldadd + col));
      }
    }
  };
  if (kPipelined) prefetch(warp_global);
  for (int row = warp_global; row < rows; row += warp_stride) {
    if (!kPipelined) {
      prefetch_l2((long long)row + warp_stride);
      prefetch(row);
    }
    const float mean = nmean, rstd = nrstd;
    float xh[NV][8], gd[NV][8];
    uint4 ca[NV];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      float d8[8];
      unpack8(nx[j], xh[j]);
      unpack8(nd[j], d8);
      if (kPipelined) ca[j] = na[j];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        xh[j][e] = (xh[j][e] - mean) * rstd;
        dgacc[j][e] += d8[e] * xh[j][e];
        gd[j][e] = d8[e] * gg[j][e];
        s1 += gd[j][e];
        s2 += gd[j][e] * xh[j][e];
      }
    }
    if (kPipelined) prefetch(row + warp_stride);
    s1 = warp_sum(s1) * (1.f / D);
    s2 = warp_sum(s2) * (1.f / D);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int col = (j * 32 + lane) * 8;
      float a8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (add != nullptr) {
        if (kPipelined) unpack8(ca[j], a8);
        else load8(add + row * ldadd + col, a8);
      }
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = rstd * (gd[j][e] - s1 - xh[j][e] * s2) + a8[e];
      store8(dx + row * lddx + col, o);
    }
  }
  if (dg != nullptr) flush_column_partials<NV>(dgacc, dg, red);
}

// ---------------------------------------------------------------------------
// l2-normalise rows of an fp32 matrix: z = p / max(||p||, 1e-12)
//   fwd writes z (fp32), the split-bf16 MMA operands zrow = [hi|lo|hi], zcol = [hi|hi|lo]
//   ([rows, 3d] each; zrow . zcol^T reproduces the fp32 dot product to ~2^-17) and
//   inv = 1/max(||p||,eps)
//   bwd: dp = inv * (dz - z * <z, dz>)   (bf16, operand of the projection dgrad/wgrad)
// ---------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kRowThreads)
l2norm_fwd_kernel(const float* __restrict__ p, long long ldp, float* __restrict__ z,
                  bf16* __restrict__ zrow, bf16* __restrict__ zcol, float* __restrict__ inv,
                  int rows) {
  const int lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  const int warp_stride = gridDim.x * kRowWarps;
  constexpr int D = NV * 256;
  for (int row = warp_global; row < rows; row += warp_stride) {
    float v[NV][8];
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      loadf8(p + row * ldp + (j * 32 + lane) * 8, v[j]);
#pragma unroll
      for (int e = 0; e < 8; ++e) q += v[j][e] * v[j][e];
    }
    const float r = 1.f / fmaxf(sqrtf(warp_sum(q)), 1e-12f);
    if (lane == 0) inv[row] = r;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int col = (j * 32 + lane) * 8;
      float hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        v[j][e] *= r;
        hi[e] = bf16_round(v[j][e]);
        lo[e] = v[j][e] - hi[e];
      }
      storef8(z + (long long)row * D + col, v[j]);
      // split-bf16 operands: <a,b> ~= a_hi.b_hi + a_lo.b_hi + a_hi.b_lo  (error ~2^-17)
      bf16* zr = zrow + (long long)row * (3 * D);
      bf16* zc = zcol + (long long)row * (3 * D);
      store8(zr + col, hi); store8(zr + D + col, lo); store8(zr + 2 * D + col, hi);
      store8(zc + col, hi); store8(zc + D + col, hi); store8(zc + 2 * D + col, lo);
    }
  }
}

template <int NV>
__global__ void __launch_bounds__(kRowThreads)
l2norm_bwd_kernel(const float* __restrict__ dz, const float* __restrict__ z,
                  const float* __restrict__ inv, bf16* __restrict__ dp, int rows) {
  const int lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  const int warp_stride = gridDim.x * kRowWarps;
  constexpr int D = NV * 256;
  for (int row = warp_global; row < rows; row += warp_stride) {
    float a[NV][8], b[NV][8];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int col = (j * 32 + lane) * 8;
      loadf8(dz + (long long)row * D + col, a[j]);
      loadf8(z + (long long)row * D + col, b[j]);
#pragma unroll
      for (int e = 0; e < 8; ++e) dot += a[j][e] * b[j][e];
    }
    dot = warp_sum(dot);
    const float r = inv[row];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int col = (j * 32 + lane) * 8;
      float o[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = r * (a[j][e] - b[j][e] * dot);
      store8(dp + (long long)row * D + col, o);
    }
  }
}

// ---------------------------------------------------------------------------
// Fused feed-forward backward helpers (see csrc/ff.cu).  The LayerNorm(4d) output h is never
// materialised; its backward only needs d-wide row quantities:
//   dxs   = bf16(dx * rstd_r)                       operand of dW2g = dxs^T hp - vsum (x) 1
//   vsum  = sum_r dxs_r * mean_r                     [d]
//   ab[r] = (a/D, rstd (t - mean a)/D),  a = <dx_r, colvec>,  t = <dx_r, acc_r>     (D = 4 d)
//           = the two row means mean_k(gdh) and mean_k(gdh * hn) of the LayerNorm backward, because
//             gdh = dx W2g and sum_k hn_k W2g_jk = (x2 - x1)_j = rstd (acc_j - mean colvec_j).
// ---------------------------------------------------------------------------
template <int NV>
__global__ void __launch_bounds__(kRowThreads, 2)
ff_bwd_prep_kernel(const bf16* __restrict__ dx, long long lddx, const float* __restrict__ stats,
                   const bf16* __restrict__ acc, long long ldacc, const float* __restrict__ colvec,
                   bf16* __restrict__ dxs, float* __restrict__ vsum, float* __restrict__ ab, int rows) {
  __shared__ float red[NV * 256];
  constexpr int D = NV * 256;
  const int lane = threadIdx.x & 31;
  const int warp_global = blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  const int warp_stride = gridDim.x * kRowWarps;
  float vacc[NV][8];
#pragma unroll
  for (int j = 0; j < NV; ++j)
#pragma unroll
    for (int e = 0; e < 8; ++e) vacc[j][e] = 0.f;
  const float invD4 = 1.f / (4.f * D);
  // Two rows per warp iteration: all 4 NV 16-byte loads of both rows are issued before anything is
  // reduced, so twice the bytes are in flight per warp and the two shuffle reductions overlap (the
  // one-row version ran at 2.5 TB/s: its warps spent most of the time in the reductions with no load
  // outstanding).  colvec is re-read from L1 instead of living in 8 NV registers.
  for (long long row0 = 2ll * warp_global; row0 < rows; row0 += 2ll * warp_stride) {
    const bool two = row0 + 1 < rows;
    uint4 rdx[2][NV], rac[2][NV];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const long long row = (r == 0 || two) ? row0 + r : row0;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const int col = (j * 32 + lane) * 8;
        rdx[r][j] = *reinterpret_cast<const uint4*>(dx + row * lddx + col);
        if (ab != nullptr) rac[r][j] = *reinterpret_cast<const uint4*>(acc + row * ldacc + col);
      }
    }
    float mean[2], rstd[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const long long row = (r == 0 || two) ? row0 + r : row0;
      mean[r] = stats[2 * row];
      rstd[r] = stats[2 * row + 1];
    }
    float a[2] = {0.f, 0.f}, t[2] = {0.f, 0.f};
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (r == 1 && !two) break;
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        const int col = (j * 32 + lane) * 8;
        float f[8];
        unpack8(rdx[r][j], f);
        if (ab != nullptr) {
          float ac[8], cv[8];
          unpack8(rac[r][j], ac);
          loadf8(colvec + col, cv);
#pragma unroll
          for (int e = 0; e < 8; ++e) { a[r] = fmaf(f[e], cv[e], a[r]); t[r] = fmaf(f[e], ac[e], t[r]); }
        }
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          o[e] = bf16_round(f[e] * rstd[r]);
          vacc[j][e] = fmaf(o[e], mean[r], vacc[j][e]);
        }
        store8(dxs + (row0 + r) * D + col, o);
      }
    }
    if (ab != nullptr) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {     // four interleaved butterfly reductions
        a[0] += __shfl_xor_sync(0xffffffffu, a[0], off);
        t[0] += __shfl_xor_sync(0xffffffffu, t[0], off);
        a[1] += __shfl_xor_sync(0xffffffffu, a[1], off);
        t[1] += __shfl_xor_sync(0xffffffffu, t[1], off);
      }
      if (lane == 0) {
        ab[2 * row0] = a[0] * invD4;
        ab[2 * row0 + 1] = rstd[0] * (t[0] - mean[0] * a[0]) * invD4;
        if (two) {
          ab[2 * row0 + 2] = a[1] * invD4;
          ab[2 * row0 + 3] = rstd[1] * (t[1] - mean[1] * a[1]) * invD4;
        }
      }
    }
  }
  flush_column_partials<NV>(vacc, vsum, red);
}

// raw = dxs^T hp (f32 [d, 4d]).  In place: dW2[j,k] = g[k] (raw[j,k] - vsum[j]);  optionally
// dg[k] += sum_j (raw[j,k] - vsum[j]) * w2[j,k]   (gain gradient of the folded LayerNorm).
// One thread per column k, blockIdx.y walks row chunks.
__global__ void __launch_bounds__(256)
ff_w2_grad_post_kernel(float* __restrict__ raw, const float* __restrict__ vsum,
                       const float* __restrict__ g, const float* __restrict__ w2,
                       float* __restrict__ dg, int d, int rows_per_block) {
  const long long D4 = 4ll * d;
  const long long k = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (k >= D4) return;
  const int j0 = blockIdx.y * rows_per_block;
  const int j1 = min(j0 + rows_per_block, d);
  const float gk = g[k];
  float acc = 0.f;
  for (int j = j0; j < j1; ++j) {
    const float t = raw[j * D4 + k] - vsum[j];
    if (w2 != nullptr) acc = fmaf(t, w2[j * D4 + k], acc);
    raw[j * D4 + k] = gk * t;
  }
  if (dg != nullptr) atomicAdd(dg + k, acc);
}

// flat fp32 -> bf16
__global__ void __launch_bounds__(256)
cast_f32_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
  const long long n8 = n / 8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8;
       i += (long long)gridDim.x * blockDim.x) {
    float f[8];
    loadf8(src + i * 8, f);
    store8(dst + i * 8, f);
  }
  if (blockIdx.x == 0 && threadIdx.x < (n & 7))
    dst[n8 * 8 + threadIdx.x] = __float2bfloat16_rn(src[n8 * 8 + threadIdx.x]);
}

static int row_grid(int rows) {
  const int blocks = (rows + kRowWarps - 1) / kRowWarps;
  const int cap = num_sms() * 8;
  return blocks < cap ? (blocks > 0 ? blocks : 1) : cap;
}

}  // namespace xclip

using namespace xclip;

#define LAUNCH_NV(KERNEL, NVAL, GRID, STREAM, ...) \
  case NVAL: KERNEL<NVAL><<<GRID, kRowThreads, 0, STREAM>>>(__VA_ARGS__); break;

#define DISPATCH_NARROW(KERNEL, D, GRID, STREAM, ...)                                     \
  switch ((D) / 256) {                                                                    \
    LAUNCH_NV(KERNEL, 1, GRID, STREAM, __VA_ARGS__)                                       \
    LAUNCH_NV(KERNEL, 2, GRID, STREAM, __VA_ARGS__)                                       \
    LAUNCH_NV(KERNEL, 3, GRID, STREAM, __VA_ARGS__)                                       \
    LAUNCH_NV(KERNEL, 4, GRID, STREAM, __VA_ARGS__)                                       \
    default:                                                                              \
      return fail(XCLIP_ERR_INVALID, "row width %d unsupported (256*{1,2,3,4})", (D));    \
  }

#define ALIGNED16(p) ((reinterpret_cast<uintptr_t>(p) & 15) == 0)

extern "C" int xclip_layernorm_fwd(const void* x, int64_t ldx, const float* g, const void* res,
                                   int64_t ldres, void* out, int64_t ldo, float* stats,
                                   const float* g2, void* out2, int64_t ldo2, float* stats2,
                                   int rows, int d, float eps, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(x && g && out, "layernorm_fwd: null pointer");
  XCLIP_REQUIRE(rows > 0, "layernorm_fwd: rows=%d", rows);
  XCLIP_REQUIRE(d % 256 == 0, "layernorm_fwd: d=%d must be a multiple of 256", d);
  XCLIP_REQUIRE(ldx % 8 == 0 && ldo % 8 == 0 && (!res || ldres % 8 == 0) && (!g2 || ldo2 % 8 == 0),
                "layernorm_fwd: leading dims must be multiples of 8");
  XCLIP_REQUIRE(ALIGNED16(x) && ALIGNED16(out) && ALIGNED16(g) && (!res || ALIGNED16(res)) &&
                    (!g2 || (ALIGNED16(g2) && out2 && ALIGNED16(out2))),
                "layernorm_fwd: pointers must be 16-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  DISPATCH_NARROW(ln_fwd_kernel, d, row_grid(rows), s, (const bf16*)x, ldx, g, (const bf16*)res,
                  ldres, (bf16*)out, ldo, stats, g2, (bf16*)out2, ldo2, stats2, rows, eps)
  XCLIP_LAUNCH_CHECK("ln_fwd_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_layernorm_bwd(const void* dy, int64_t lddy, const void* x, int64_t ldx,
                                   const float* stats, const float* g, const void* add,
                                   int64_t ldadd, void* dx, int64_t lddx, float* dg, int rows,
                                   int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(dy && x && stats && g && dx, "layernorm_bwd: null pointer");
  XCLIP_REQUIRE(rows > 0 && d % 256 == 0, "layernorm_bwd: rows=%d d=%d", rows, d);
  XCLIP_REQUIRE(lddy % 8 == 0 && ldx % 8 == 0 && lddx % 8 == 0 && (!add || ldadd % 8 == 0),
                "layernorm_bwd: leading dims must be multiples of 8");
  XCLIP_REQUIRE(ALIGNED16(dy) && ALIGNED16(x) && ALIGNED16(dx) && ALIGNED16(g) &&
                    (!add || ALIGNED16(add)),
                "layernorm_bwd: pointers must be 16-byte aligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int per_sm = 2;
  const int grid = row_grid(rows) < num_sms() * per_sm ? row_grid(rows) : num_sms() * per_sm;
  DISPATCH_NARROW(ln_bwd_kernel, d, grid, s, (const bf16*)dy, lddy, (const bf16*)x, ldx, stats, g,
                  (const bf16*)add, ldadd, (bf16*)dx, lddx, dg, rows)
  XCLIP_LAUNCH_CHECK("ln_bwd_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_l2norm_fwd(const float* p, int64_t ldp, float* z, void* zrow, void* zcol,
                                float* inv, int rows, int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(p && z && zrow && zcol && inv, "l2norm_fwd: null pointer");
  XCLIP_REQUIRE(rows > 0 && d % 256 == 0, "l2norm_fwd: rows=%d d=%d", rows, d);
  XCLIP_REQUIRE(ldp % 4 == 0 && ALIGNED16(p) && ALIGNED16(z) && ALIGNED16(zrow) && ALIGNED16(zcol),
                "l2norm_fwd: misaligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  DISPATCH_NARROW(l2norm_fwd_kernel, d, row_grid(rows), s, p, ldp, z, (bf16*)zrow, (bf16*)zcol,
                  inv, rows)
  XCLIP_LAUNCH_CHECK("l2norm_fwd_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_l2norm_bwd(const float* dz, const float* z, const float* inv, void* dp,
                                int rows, int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(dz && z && inv && dp, "l2norm_bwd: null pointer");
  XCLIP_REQUIRE(rows > 0 && d % 256 == 0, "l2norm_bwd: rows=%d d=%d", rows, d);
  XCLIP_REQUIRE(ALIGNED16(dz) && ALIGNED16(z) && ALIGNED16(dp), "l2norm_bwd: misaligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  DISPATCH_NARROW(l2norm_bwd_kernel, d, row_grid(rows), s, dz, z, inv, (bf16*)dp, rows)
  XCLIP_LAUNCH_CHECK("l2norm_bwd_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_cast_f32_bf16(const float* src, void* dst, int64_t n, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(src && dst && n > 0, "cast: bad arguments");
  XCLIP_REQUIRE(ALIGNED16(src) && ALIGNED16(dst), "cast: misaligned");
  long long blocks = (n / 8 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > num_sms() * 8) blocks = num_sms() * 8;
  cast_f32_bf16_kernel<<<(int)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      src, (bf16*)dst, n);
  XCLIP_LAUNCH_CHECK("cast_f32_bf16_kernel");
  return XCLIP_OK;
}

// ---------------------------------------------------------------------------
// Fused AdamW over one flat fp32 buffer (SURVEY 8f rank 2: the optimizer step behind the
// weight-gradient all-reduce).  Same update as torch.optim.AdamW (decoupled weight decay):
//   p *= 1 - lr*wd;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)          g = grad * grad_scale
// 7 streams of 4 bytes per element: HBM-bound.
// ---------------------------------------------------------------------------
namespace xclip {
__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
             float* __restrict__ v, long long n4, long long n, float lr, float b1, float b2, float eps,
             float decay, float step_size, float inv_sqrt_bc2, float gscale) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    const float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pe = reinterpret_cast<float*>(&pp);
    const float* ge = reinterpret_cast<const float*>(&gg);
    float* me = reinterpret_cast<float*>(&mm);
    float* ve = reinterpret_cast<float*>(&vv);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float gr = ge[e] * gscale;
      me[e] = b1 * me[e] + (1.f - b1) * gr;
      ve[e] = b2 * ve[e] + (1.f - b2) * gr * gr;
      const float denom = sqrtf(ve[e]) * inv_sqrt_bc2 + eps;
      pe[e] = pe[e] * decay - step_size * (me[e] / denom);
    }
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  // tail (n not a multiple of 4)
  const long long i = n4 * 4 + blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) {
    const float gr = g[i] * gscale;
    const float mn = b1 * m[i] + (1.f - b1) * gr;
    const float vn = b2 * v[i] + (1.f - b2) * gr * gr;
    m[i] = mn; v[i] = vn;
    p[i] = p[i] * decay - step_size * (mn / (sqrtf(vn) * inv_sqrt_bc2 + eps));
  }
}
}  // namespace xclip

extern "C" int xclip_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr,
                                float beta1, float beta2, float eps, float weight_decay, int step,
                                float grad_scale, xclip_stream_t stream) {
  using namespace xclip;
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(p && g && m && v && n > 0 && step >= 1, "adamw: bad arguments");
  XCLIP_REQUIRE(ALIGNED16(p) && ALIGNED16(g) && ALIGNED16(m) && ALIGNED16(v), "adamw: buffers must be 16-byte aligned");
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  const long long n4 = n / 4;
  long long blocks = (n4 + 255) / 256;
  if (blocks > (long long)num_sms() * 16) blocks = (long long)num_sms() * 16;
  if (blocks < 1) blocks = 1;
  adamw_kernel<<<(int)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      p, g, m, v, n4, n, lr, beta1, beta2, eps, 1.f - lr * weight_decay, (float)(lr / bc1),
      (float)(1.0 / sqrt(bc2)), grad_scale);
  XCLIP_LAUNCH_CHECK("adamw_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_ff_bwd_prep(const void* dx, int64_t lddx, const float* stats, const void* acc,
                                 int64_t ldacc, const float* colvec, void* dxs, float* vsum, float* ab,
                                 int rows, int d, xclip_stream_t stream) {
  using namespace xclip;
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(dx && stats && dxs && vsum && rows > 0, "ff_bwd_prep: bad arguments");
  XCLIP_REQUIRE(d % 256 == 0, "ff_bwd_prep: d=%d must be a multiple of 256", d);
  XCLIP_REQUIRE(ab == nullptr || (acc && colvec), "ff_bwd_prep: ab needs acc and colvec");
  XCLIP_REQUIRE(lddx % 8 == 0 && lddx >= d && ALIGNED16(dx) && ALIGNED16(dxs) &&
                    (!acc || (ALIGNED16(acc) && ldacc % 8 == 0 && ldacc >= d)) && (!colvec || ALIGNED16(colvec)),
                "ff_bwd_prep: misaligned");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int grid = row_grid(rows) < num_sms() * 4 ? row_grid(rows) : num_sms() * 4;
  DISPATCH_NARROW(ff_bwd_prep_kernel, d, grid, s, (const bf16*)dx, lddx, stats, (const bf16*)acc, ldacc,
                  colvec, (bf16*)dxs, vsum, ab, rows)
  XCLIP_LAUNCH_CHECK("ff_bwd_prep_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_ff_w2_grad_post(float* raw, const float* vsum, const float* g, const float* w2,
                                     float* dg, int d, xclip_stream_t stream) {
  using namespace xclip;
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(raw && vsum && g && d > 0 && d % 256 == 0, "ff_w2_grad_post: bad arguments");
  XCLIP_REQUIRE((dg == nullptr) == (w2 == nullptr), "ff_w2_grad_post: dg and w2 go together");
  const int rows_per_block = 8;      // 4d/256 x d/8 blocks: enough loads in flight for a 28 MB pass
  dim3 grid((4 * d + 255) / 256, (d + rows_per_block - 1) / rows_per_block);
  ff_w2_grad_post_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(raw, vsum, g, w2, dg, d,
                                                                                 rows_per_block);
  XCLIP_LAUNCH_CHECK("ff_w2_grad_post_kernel");
  return XCLIP_OK;
}
