// Fused feed-forward block (reference x_clip/x_clip.py:180-199) on the CTA-pair GEMM:
//   u = xn W1^T, hp = value * gelu(gate)          one GEMM, GEGLU in its epilogue   (xclip_ff_up)
//   x2 = LN_4d(hp) g W2^T + x1                     one GEMM, LayerNorm folded into
//                                                  weight + epilogue                (xclip_ff_down)
// so the [tokens, 8d] / [tokens, 4d] hidden activations make no extra round trip through HBM for
// the activation and the normalisation (a separate GEGLU + LayerNorm pass was 10 % of the cfg3 step
// and instruction-issue bound).  The LayerNorm fold:
//   LN(hp)_k g_k = (hp_k - mean) rstd g_k   =>   x2_j = rstd (sum_k hp_k W2g_jk - mean c_j),
//   W2g = W2 . g (column scaling), c_j = sum_k W2g_jk.
// Backward pieces that replace the LayerNorm output h (never materialised now):
//   dW2_jk = g_k (sum_r dxs_rj hp_rk - v_j),  dxs = dx * rstd_r,  v_j = sum_r dxs_rj mean_r
// (xclip_ff_bwd_prep, xclip_ff_w2_grad_post); everything else of the backward is unchanged.
#include "gemm_pair.cuh"
#include "host.h"

namespace xclip {

// out[256 t + i] = w1[128 t + i] (i < 128: value rows) | w1[4d + 128 t + i - 128] (gate rows)
__global__ void __launch_bounds__(256)
ff_permute_cast_kernel(const float* __restrict__ w1, bf16* __restrict__ out, int d) {
  const long long vec_per_row = d / 8;
  const long long total = 8ll * d * vec_per_row;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long orow = idx / vec_per_row;
    const int c = (int)(idx - orow * vec_per_row) * 8;
    const long long t = orow >> 8;
    const int i = (int)(orow & 255);
    const long long srow = i < 128 ? 128 * t + i : 4ll * d + 128 * t + (i - 128);
    const float4 a = *reinterpret_cast<const float4*>(w1 + srow * d + c);
    const float4 b = *reinterpret_cast<const float4*>(w1 + srow * d + c + 4);
    uint4 o;
    o.x = pack_bf16x2(a.x, a.y); o.y = pack_bf16x2(a.z, a.w);
    o.z = pack_bf16x2(b.x, b.y); o.w = pack_bf16x2(b.z, b.w);
    *reinterpret_cast<uint4*>(out + orow * d + c) = o;
  }
}

// w2g[j,k] = bf16(w2[j,k] * g[k]);  colvec[j] = sum_k float(w2g[j,k]).   One block per row j.
__global__ void __launch_bounds__(256)
ff_scale_cast_kernel(const float* __restrict__ w2, const float* __restrict__ g, bf16* __restrict__ w2g,
                     float* __restrict__ colvec, int d) {
  __shared__ float red[8];
  const int j = blockIdx.x;
  const long long D = 4ll * d;
  float s = 0.f;
  for (long long k = threadIdx.x * 8; k < D; k += 256 * 8) {
    const float4 a = *reinterpret_cast<const float4*>(w2 + j * D + k);
    const float4 b = *reinterpret_cast<const float4*>(w2 + j * D + k + 4);
    const float4 ga = *reinterpret_cast<const float4*>(g + k);
    const float4 gb = *reinterpret_cast<const float4*>(g + k + 4);
    const float f[8] = {a.x * ga.x, a.y * ga.y, a.z * ga.z, a.w * ga.w,
                        b.x * gb.x, b.y * gb.y, b.z * gb.z, b.w * gb.w};
    uint4 o;
    o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
    o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(w2g + j * D + k) = o;
#pragma unroll
    for (int e = 0; e < 8; ++e) s += bf16_rn(f[e]);
  }
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < 8; ++w) tot += red[w];
    colvec[j] = tot;
  }
}

template <int EPI, int B_MAJOR = kMajorK>
static int launch_pair_ff(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC,
                          const CUtensorMap& tmC2, const GemmParams& p, cudaStream_t stream) {
  using S = PairCfg<EPI>;
  auto kern = gemm_pair_kernel<kMajorK, B_MAJOR, EPI>;
  const int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), S::kTotal);
  if (rc) return rc;
  const long long tiles = (long long)((p.M + 255) / 256) * ((p.N + 255) / 256);
  const int units = num_sms() / 2;
  const int pairs = (int)(tiles < units ? tiles : units);
  kern<<<2 * pairs, S::kThreads, S::kTotal, stream>>>(tmA, tmB, tmC, tmC2, p);
  XCLIP_LAUNCH_CHECK("gemm_pair_kernel<ff>");
  return XCLIP_OK;
}

}  // namespace xclip

using namespace xclip;

#define FF_ALIGNED(p) ((reinterpret_cast<uintptr_t>(p) & 15) == 0)

extern "C" int xclip_ff_permute_cast(const float* w1, void* out, int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(w1 && out && d > 0 && d % 256 == 0, "ff_permute_cast: d=%d must be a multiple of 256", d);
  XCLIP_REQUIRE(FF_ALIGNED(w1) && FF_ALIGNED(out), "ff_permute_cast: misaligned pointer");
  ff_permute_cast_kernel<<<num_sms() * 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      w1, reinterpret_cast<bf16*>(out), d);
  XCLIP_LAUNCH_CHECK("ff_permute_cast_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_ff_scale_cast(const float* w2, const float* g, void* w2g, float* colvec, int d,
                                   xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(w2 && g && w2g && colvec && d > 0 && d % 256 == 0, "ff_scale_cast: bad arguments");
  XCLIP_REQUIRE(FF_ALIGNED(w2) && FF_ALIGNED(g) && FF_ALIGNED(w2g), "ff_scale_cast: misaligned pointer");
  ff_scale_cast_kernel<<<d, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      w2, g, reinterpret_cast<bf16*>(w2g), colvec, d);
  XCLIP_LAUNCH_CHECK("ff_scale_cast_kernel");
  return XCLIP_OK;
}

extern "C" int xclip_ff_up(const void* x, int64_t ldx, const void* w1p, void* u, int64_t ldu, void* hp,
                           int64_t ldhp, float* rowsum, int M, int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(x && w1p && hp && rowsum, "ff_up: null pointer");
  const bool skip_u = (u == nullptr);      // forward-only sweeps: hp is all the down-projection needs
  if (skip_u) { u = hp; ldu = ldhp >= 8 * (int64_t)d ? ldhp : 8 * (int64_t)d; }   // (placeholder map, never stored to)
  XCLIP_REQUIRE(M > 0 && d > 0 && d % 256 == 0, "ff_up: M=%d d=%d (d %% 256)", M, d);
  XCLIP_REQUIRE(ldx % 8 == 0 && ldx >= d && ldu % 8 == 0 && ldu >= 8 * d && ldhp % 8 == 0 && ldhp >= 4 * d,
                "ff_up: bad leading dimensions");
  XCLIP_REQUIRE(FF_ALIGNED(x) && FF_ALIGNED(w1p) && FF_ALIGNED(u) && FF_ALIGNED(hp), "ff_up: misaligned pointer");
  CUtensorMap tmA, tmB, tmC, tmC2;
  if ((rc = encode_2d_bf16(&tmA, x, (uint64_t)d, (uint64_t)M, (uint64_t)ldx, 64, kGemmBlockM))) return rc;
  if ((rc = encode_2d_bf16(&tmB, w1p, (uint64_t)d, (uint64_t)(8 * d), (uint64_t)d, 64, 128))) return rc;
  if (skip_u) {
    if ((rc = encode_2d_bf16(&tmC, hp, (uint64_t)(4 * d), (uint64_t)M, (uint64_t)ldhp, 64, kGemmBlockM))) return rc;
  } else if ((rc = encode_2d_bf16(&tmC, u, (uint64_t)(8 * d), (uint64_t)M, (uint64_t)ldu, 64, kGemmBlockM))) return rc;
  if ((rc = encode_2d_bf16(&tmC2, hp, (uint64_t)(4 * d), (uint64_t)M, (uint64_t)ldhp, 64, kGemmBlockM))) return rc;
  GemmParams p = {};
  p.M = M; p.N = 8 * d; p.K = d; p.split_k = 1; p.alpha = 1.f;
  p.ff_rowsum = rowsum; p.ff_hidden = 4 * d; p.ff_skip_u = skip_u ? 1 : 0;
  return launch_pair_ff<PEPI_FF_UP>(tmA, tmB, tmC, tmC2, p, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int xclip_ff_down(const void* hp, int64_t ldhp, const void* w2g, const float* colvec,
                             const float* rowsum, const void* residual, int64_t ldr, void* out,
                             int64_t ldo, void* acc_out, int64_t ldacc, float* stats, float eps, int M,
                             int d, xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(hp && w2g && colvec && rowsum && out && acc_out && stats, "ff_down: null pointer");
  XCLIP_REQUIRE(M > 0 && d > 0 && d % 256 == 0, "ff_down: M=%d d=%d (d %% 256)", M, d);
  XCLIP_REQUIRE(ldhp % 8 == 0 && ldhp >= 4 * d && ldo % 8 == 0 && ldo >= d && ldacc % 8 == 0 && ldacc >= d &&
                    (!residual || (ldr % 8 == 0 && ldr >= d)),
                "ff_down: bad leading dimensions");
  XCLIP_REQUIRE(FF_ALIGNED(hp) && FF_ALIGNED(w2g) && FF_ALIGNED(out) && FF_ALIGNED(acc_out) &&
                    FF_ALIGNED(colvec) && (!residual || FF_ALIGNED(residual)),
                "ff_down: misaligned pointer");
  CUtensorMap tmA, tmB, tmC, tmC2;
  if ((rc = encode_2d_bf16(&tmA, hp, (uint64_t)(4 * d), (uint64_t)M, (uint64_t)ldhp, 64, kGemmBlockM))) return rc;
  if ((rc = encode_2d_bf16(&tmB, w2g, (uint64_t)(4 * d), (uint64_t)d, (uint64_t)(4 * d), 64, 128))) return rc;
  if ((rc = encode_2d_bf16(&tmC, out, (uint64_t)d, (uint64_t)M, (uint64_t)ldo, 64, kGemmBlockM))) return rc;
  if ((rc = encode_2d_bf16(&tmC2, acc_out, (uint64_t)d, (uint64_t)M, (uint64_t)ldacc, 64, kGemmBlockM))) return rc;
  GemmParams p = {};
  p.M = M; p.N = d; p.K = 4 * d; p.split_k = 1; p.alpha = 1.f;
  p.residual = reinterpret_cast<const bf16*>(residual); p.ldr = ldr;
  p.ff_rowsum = const_cast<float*>(rowsum); p.ff_colvec = colvec; p.ff_stats = stats;
  p.ff_eps = eps; p.ff_hidden = 4 * d;
  return launch_pair_ff<PEPI_FF_DOWN>(tmA, tmB, tmC, tmC2, p, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int xclip_ff_bwd(const void* dx, int64_t lddx, const void* w2g, const void* u, int64_t ldu,
                            const float* stats, const float* ab, void* du, int64_t lddu, int M, int d,
                            xclip_stream_t stream) {
  int rc = xclip_init();
  if (rc) return rc;
  XCLIP_REQUIRE(dx && w2g && u && stats && ab && du, "ff_bwd: null pointer");
  XCLIP_REQUIRE(M > 0 && d > 0 && d % 256 == 0, "ff_bwd: M=%d d=%d (d %% 256)", M, d);
  XCLIP_REQUIRE(lddx % 8 == 0 && lddx >= d && ldu % 8 == 0 && ldu >= 8 * d && lddu % 8 == 0 && lddu >= 8 * d,
                "ff_bwd: bad leading dimensions");
  XCLIP_REQUIRE(FF_ALIGNED(dx) && FF_ALIGNED(w2g) && FF_ALIGNED(u) && FF_ALIGNED(du), "ff_bwd: misaligned pointer");
  CUtensorMap tmA, tmB, tmC;
  if ((rc = encode_2d_bf16(&tmA, dx, (uint64_t)d, (uint64_t)M, (uint64_t)lddx, 64, kGemmBlockM))) return rc;
  // B = w2g [d, 4d] consumed MN-major: contraction index d on rows, 64 x 64 boxes
  if ((rc = encode_2d_bf16(&tmB, w2g, (uint64_t)(4 * d), (uint64_t)d, (uint64_t)(4 * d), 64, kGemmBlockK))) return rc;
  if ((rc = encode_2d_bf16(&tmC, du, (uint64_t)(8 * d), (uint64_t)M, (uint64_t)lddu, 64, kGemmBlockM))) return rc;
  GemmParams p = {};
  p.M = M; p.N = 4 * d; p.K = d; p.split_k = 1; p.alpha = 1.f;
  p.ff_stats = const_cast<float*>(stats); p.ff_ab = ab; p.ff_hidden = 4 * d;
  CUtensorMap tmU;                               // u = [value | gate], loaded box-wise ahead of its step
  if ((rc = encode_2d_bf16(&tmU, u, (uint64_t)(8 * d), (uint64_t)M, (uint64_t)ldu, 64, kGemmBlockM))) return rc;
  return launch_pair_ff<PEPI_FF_BWD2, kMajorMN>(tmA, tmB, tmC, tmU, p, reinterpret_cast<cudaStream_t>(stream));
}
