// Persistent, warp-specialised tcgen05 GEMM for sm_100a.
//
//   C[M,N] = alpha * A * B^T (+ bias[N]) (+ residual[M,N])        bf16 x bf16 -> fp32 accum
//
// Operand storage (both cases are fed straight from global memory by TMA, no transposes):
//   a_major = K  : A is [M,K] row-major (K contiguous)          - activations in fwd / dgrad
//   a_major = MN : A is given as At[K,M] row-major (M contiguous)- dY^T in wgrad
//   b_major = K  : B is [N,K] row-major                          - nn.Linear weight [out,in] in fwd
//   b_major = MN : B is given as Bt[K,N] row-major (N contiguous)- weight in dgrad, X in wgrad
//
// This one kernel covers the reference's nn.Linear call sites on the hot path
// (x_clip/x_clip.py:191,195,209,210,358,368,556,570) and their autograd backward.
//
// Structure (one CTA per SM, 192 threads):
//   warps 0-3 : epilogue  (TMEM -> registers -> global; warp w owns TMEM lanes 32w..32w+31)
//   warp  4   : TMA producer (one elected lane)
//   warp  5   : TMEM allocator + MMA issuer (one lane issues tcgen05.mma / tcgen05.commit)
// Pipelines: smem ring full/empty (TMA <-> MMA), TMEM accumulators double-buffered
// full/empty (MMA <-> epilogue), static persistent tile scheduler with optional split-K.
#pragma once

#include "common.cuh"

namespace xclip {

struct GemmParams {
  int M, N, K;
  void* c;
  long long ldc;
  int c_is_f32;        // 0: bf16 out, 1: fp32 out
  int atomic_add;      // fp32 out only: red.add into C (required when split_k > 1)
  int split_k;
  float alpha;
  const float* bias;   // [N] or null
  const bf16* residual;  // bf16 [*, N] or null
  long long ldr;
  int res_row_mod;     // residual row = row % res_row_mod when > 0 (positional tables)
  const int* res_row_idx;  // or residual row = res_row_idx[row] (gathered positional rows), else row
  int use_tma_store;   // bf16 C written through swizzled smem staging + cp.async.bulk.tensor stores
  int raster_m_fast;   // tile order: 0 = N fastest (big A streamed once, B tile L2 resident),
                       //             1 = M fastest (small A resident, big B streamed once)
  // ---- InfoNCE / DCL epilogues (EPI_NCE_FWD, EPI_NCE_BWD); logits s = alpha * acc, alpha = exp(temperature)
  int diag_offset;       // positive of local row r sits in column r + diag_offset
  int dcl;               // decoupled contrastive learning: drop the positive from the denominators
  float* nce_part;       // FWD: [num_n_blocks, M, 2] per block (max of x, sum of 2^(x - max)), x = s*log2(e)
  float* nce_pos;        // FWD: [M] positive logits
  const float* lse_row;  // BWD: [M]  log-denominator of each row (this direction)
  const float* lse_col;  // BWD: [N]  log-denominator of each column (other direction)
  float w_row, w_col, w_diag;
  float* dtemp;          // BWD: scalar accumulator of sum(g * s) or null
  const float* alpha_dev;  // NCE: exp(temperature) read from device memory (no host sync)
  const float* gscale_dev; // BWD: upstream scalar gradient / (2*B_global), multiplies the weights
  // ---- FILIP segment-max epilogue (EPI_SEGMAX): columns are grouped in segments of seg_len
  // tokens (one segment = one sample of the other modality); n_tile_stride = columns a tile
  // advances by (a whole number of segments, <= BLOCK_N)
  int seg_len, n_tile_stride, n_segs;
  const float* col_mul;    // [N] or null: per-column multiplier (0 for masked text tokens)
  const float* col_add;    // [N] or null: per-column addend (-FLT_MAX for masked text tokens)
  float* seg_max;          // [M, n_segs]  max_i s
  int* seg_arg;            // [M, n_segs]  argmax (index inside the segment)
  // ---- fused feed-forward epilogues of the CTA-pair kernel (gemm_pair.cuh)
  float* ff_rowsum;        // [M, 4d/64, 2] per-box (sum, sum of squares) of the GEGLU output rows: UP writes, DOWN sums
  const float* ff_colvec;  // DOWN: c[N] = row sums of the gain-scaled down-projection weight
  float* ff_stats;         // DOWN: [M,2] (mean, rstd) of the GEGLU output rows, written for the backward
  float ff_eps;            // LayerNorm epsilon
  int ff_hidden;           // 4*dim: LayerNorm width; column offset of the gate half inside u
  int ff_skip_u;           // UP: do not write u = [value | gate] (inference / no-grad sweeps need only hp)
  const float* ff_ab;      // BWD: [M,2] per-row (mean_k(gdh), mean_k(gdh * hn)) from xclip_ff_bwd_prep
};

constexpr int EPI_STORE = 0;    // C = alpha*acc (+bias) (+residual)
constexpr int EPI_NCE_FWD = 1;  // row partial sums of exp(s - alpha) and the positives
constexpr int EPI_NCE_BWD = 2;  // C = g = w_row*exp(s-lse_row) + w_col*exp(s-lse_col) - w_diag*[diag]
constexpr int EPI_SEGMAX = 3;   // per row and column segment: max and argmax of alpha*acc (FILIP)

constexpr int kGemmBlockM = 128;
constexpr int kGemmBlockK = 64;
constexpr int kGemmThreads = 192;

template <int BLOCK_N>
struct GemmSmem {
  static constexpr int kABytes = kGemmBlockM * kGemmBlockK * 2;  // 16 KiB
  static constexpr int kBBytes = BLOCK_N * kGemmBlockK * 2;      // 16/32 KiB
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BLOCK_N == 256) ? 4 : 6;
  static constexpr int kBarrierBytes = 256;
  static constexpr int kStagingBytes = 2 * 128 * 128;  // two [128 rows x 64 bf16] output boxes
  static constexpr int kTotal = kStages * kStageBytes + kStagingBytes + kBarrierBytes;
};

__device__ __forceinline__ float nce_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Epilogue of one 128 x BLOCK_N accumulator tile (EPI_STORE): C = alpha*acc (+bias) (+residual) as
// bf16 through swizzled smem staging + TMA stores, or fp32 direct / atomic.  Called by the four
// epilogue warps (warp = 0..3 owns TMEM lanes 32*warp..+31); `store_count` is the running parity of
// the two staging buffers.
template <int BLOCK_N>
__device__ __forceinline__ void gemm_epilogue_store(const GemmParams& p, const CUtensorMap& tmC,
                                                    uint8_t* smem_c, uint32_t taddr, int warp,
                                                    int lane, int m_blk, int n_blk, int split,
                                                    uint32_t& store_count) {
  const int row = m_blk * kGemmBlockM + warp * 32 + lane;
  const bool row_ok = row < p.M;
  const bf16* res_row = nullptr;
  if (p.residual != nullptr && row_ok) {
    const long long rr = p.res_row_idx ? p.res_row_idx[row] : (p.res_row_mod > 0 ? (row % p.res_row_mod) : row);
    res_row = p.residual + rr * p.ldr;
  }
        if (p.use_tma_store) {
          // bf16 output: 64-column boxes staged in swizzled smem (double buffered), written by
          // cp.async.bulk.tensor stores (full-line writes, no LSU pressure, tails clipped by TMA)
          const int row_in_tile = warp * 32 + lane;
#pragma unroll 1
          for (int q = 0; q < BLOCK_N / 64; ++q) {
            const uint32_t stg = smem_u32(smem_c) + (store_count & 1) * 16384;
            if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
            for (int c32 = 0; c32 < 2; ++c32) {
              uint32_t v[32];
              tmem_ld_32x32(taddr + q * 64 + c32 * 32, v);
              tmem_ld_wait();
              const int col0 = n_blk * BLOCK_N + q * 64 + c32 * 32;
              float f[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]) * p.alpha;
              if (p.bias != nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  if (col0 + i < p.N) {
                    const float4 b4 = *reinterpret_cast<const float4*>(p.bias + col0 + i);
                    f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
                  }
                }
              }
              if (res_row != nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 8) {
                  if (col0 + i < p.N) {
                    const uint4 r4 = *reinterpret_cast<const uint4*>(res_row + col0 + i);
                    float2 a = unpack_bf16x2(r4.x), b = unpack_bf16x2(r4.y);
                    float2 cc = unpack_bf16x2(r4.z), d = unpack_bf16x2(r4.w);
                    f[i] += a.x; f[i + 1] += a.y; f[i + 2] += b.x; f[i + 3] += b.y;
                    f[i + 4] += cc.x; f[i + 5] += cc.y; f[i + 6] += d.x; f[i + 7] += d.y;
                  }
                }
              }
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(
                                 stg + swz128(row_in_tile, c32 * 4 + i)),
                             "r"(pack_bf16x2(f[i * 8 + 0], f[i * 8 + 1])),
                             "r"(pack_bf16x2(f[i * 8 + 2], f[i * 8 + 3])),
                             "r"(pack_bf16x2(f[i * 8 + 4], f[i * 8 + 5])),
                             "r"(pack_bf16x2(f[i * 8 + 6], f[i * 8 + 7]))
                             : "memory");
              }
            }
            fence_proxy_async_smem();
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (threadIdx.x == 0) {
              const int c0 = n_blk * BLOCK_N + q * 64;
              if (c0 < p.N) {
                asm volatile(
                    "cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                        reinterpret_cast<uint64_t>(&tmC)),
                    "r"(stg), "r"(c0), "r"(m_blk * kGemmBlockM)
                    : "memory");
              }
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            ++store_count;
          }
        } else {
  #pragma unroll 1
        for (int c = 0; c < BLOCK_N / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
          const int col0 = n_blk * BLOCK_N + c * 32;
          if (row_ok && col0 < p.N) {
            float f[32];
  #pragma unroll
            for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]) * p.alpha;
            if (p.bias != nullptr && split == 0) {
  #pragma unroll
              for (int i = 0; i < 32; i += 4) {
                if (col0 + i < p.N) {
                  const float4 b4 = *reinterpret_cast<const float4*>(p.bias + col0 + i);
                  f[i] += b4.x; f[i + 1] += b4.y; f[i + 2] += b4.z; f[i + 3] += b4.w;
                }
              }
            }
            if (res_row != nullptr && split == 0) {
  #pragma unroll
              for (int i = 0; i < 32; i += 8) {
                if (col0 + i < p.N) {
                  const uint4 r4 = *reinterpret_cast<const uint4*>(res_row + col0 + i);
                  float2 a = unpack_bf16x2(r4.x), b = unpack_bf16x2(r4.y);
                  float2 cc = unpack_bf16x2(r4.z), d = unpack_bf16x2(r4.w);
                  f[i] += a.x; f[i + 1] += a.y; f[i + 2] += b.x; f[i + 3] += b.y;
                  f[i + 4] += cc.x; f[i + 5] += cc.y; f[i + 6] += d.x; f[i + 7] += d.y;
                }
              }
            }
            if (p.c_is_f32) {
              float* crow = reinterpret_cast<float*>(p.c) + static_cast<long long>(row) * p.ldc + col0;
              if (p.atomic_add) {
  #pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  if (col0 + i < p.N) {
                    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(crow + i),
                                 "f"(f[i]), "f"(f[i + 1]), "f"(f[i + 2]), "f"(f[i + 3])
                                 : "memory");
                  }
                }
              } else {
  #pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  if (col0 + i < p.N)
                    *reinterpret_cast<float4*>(crow + i) =
                        make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
                }
              }
            } else {
              bf16* crow = reinterpret_cast<bf16*>(p.c) + static_cast<long long>(row) * p.ldc + col0;
  #pragma unroll
              for (int i = 0; i < 32; i += 8) {
                if (col0 + i < p.N) {
                  uint4 o;
                  o.x = pack_bf16x2(f[i], f[i + 1]);
                  o.y = pack_bf16x2(f[i + 2], f[i + 3]);
                  o.z = pack_bf16x2(f[i + 4], f[i + 5]);
                  o.w = pack_bf16x2(f[i + 6], f[i + 7]);
                  *reinterpret_cast<uint4*>(crow + i) = o;
                }
              }
            }
          }
        }
        }
}

template <int BLOCK_N, int A_MAJOR, int B_MAJOR, int EPI = EPI_STORE>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const GemmParams p) {
  using S = GemmSmem<BLOCK_N>;
  constexpr int kStages = S::kStages;
  constexpr uint32_t kTmemCols = 2 * BLOCK_N;  // double-buffered accumulator
  static_assert(kTmemCols == 256 || kTmemCols == 512, "BLOCK_N must be 128 or 256");

  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * S::kABytes;
  uint8_t* smem_c = smem + kStages * S::kStageBytes;     // epilogue staging (TMA store source)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + S::kStagingBytes);
  uint64_t* full_bar = bars;                    // [kStages]
  uint64_t* empty_bar = bars + kStages;         // [kStages]
  uint64_t* tmem_full = bars + 2 * kStages;     // [2]
  uint64_t* tmem_empty = bars + 2 * kStages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int num_m = (p.M + kGemmBlockM - 1) / kGemmBlockM;
  const int n_stride = (EPI == EPI_SEGMAX) ? p.n_tile_stride : BLOCK_N;
  const int num_n = (p.N + n_stride - 1) / n_stride;
  const int num_kb = (p.K + kGemmBlockK - 1) / kGemmBlockK;
  const int splits = p.split_k > 0 ? p.split_k : 1;
  const int kb_per_split = (num_kb + splits - 1) / splits;
  const int num_tiles = num_m * num_n * splits;

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) {
      printf("xclip gemm: dynamic shared memory is not 1024-byte aligned\n");
      __trap();
    }
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 4 && XCLIP_ONE_LANE(lane)) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.use_tma_store || EPI == EPI_NCE_BWD) tma_prefetch_desc(&tmC);
  }
  if (warp == 5) tmem_alloc<kTmemCols>(tmem_slot);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ===================== TMA producer =====================
    if (XCLIP_ONE_LANE(lane)) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int tmn = t % (num_n * num_m);
        const int n_blk = p.raster_m_fast ? tmn / num_m : tmn % num_n;
        const int m_blk = p.raster_m_fast ? tmn % num_m : tmn / num_n;
        const int split = t / (num_n * num_m);
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, num_kb);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          mbar_arrive_expect_tx(&full_bar[stage], S::kStageBytes);
          uint8_t* sa = smem_a + stage * S::kABytes;
          uint8_t* sb = smem_b + stage * S::kBBytes;
          if (A_MAJOR == kMajorK) {
            tma_load_2d(sa, &tmA, &full_bar[stage], kb * kGemmBlockK, m_blk * kGemmBlockM);
          } else {
#pragma unroll
            for (int g = 0; g < kGemmBlockM / 64; ++g)
              tma_load_2d(sa + g * (kGemmBlockK * 128), &tmA, &full_bar[stage],
                          m_blk * kGemmBlockM + g * 64, kb * kGemmBlockK);
          }
          if (B_MAJOR == kMajorK) {
            tma_load_2d(sb, &tmB, &full_bar[stage], kb * kGemmBlockK, n_blk * n_stride);
          } else {
#pragma unroll
            for (int g = 0; g < BLOCK_N / 64; ++g)
              tma_load_2d(sb + g * (kGemmBlockK * 128), &tmB, &full_bar[stage],
                          n_blk * n_stride + g * 64, kb * kGemmBlockK);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = make_idesc_bf16(kGemmBlockM, BLOCK_N, A_MAJOR, B_MAJOR);
    // K-major: SBO = 1024 (8 rows x 128 B), LBO unused.  MN-major: SBO = 1024 between
    // 8-row K groups, LBO = BLOCK_K*128 between 64-wide M/N groups (one TMA box each).
    constexpr uint32_t kLboMN = kGemmBlockK * 128;
    constexpr uint32_t kAStep = (A_MAJOR == kMajorK) ? 32u : 2048u;  // bytes per UMMA_K=16
    constexpr uint32_t kBStep = (B_MAJOR == kMajorK) ? 32u : 2048u;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int split = t / (num_n * num_m);
      const int kb0 = split * kb_per_split;
      const int kb1 = min(kb0 + kb_per_split, num_kb);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tcgen05_fence_after();
      const uint32_t tmem_d = tmem_base + acc * BLOCK_N;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tcgen05_fence_after();
        if (XCLIP_ONE_LANE(lane)) {
          const uint32_t a_addr = smem_u32(smem_a + stage * S::kABytes);
          const uint32_t b_addr = smem_u32(smem_b + stage * S::kBBytes);
          const uint64_t adesc =
              make_smem_desc(a_addr, A_MAJOR == kMajorK ? 0u : kLboMN, 1024u);
          const uint64_t bdesc =
              make_smem_desc(b_addr, B_MAJOR == kMajorK ? 0u : kLboMN, 1024u);
#pragma unroll
          for (int k = 0; k < kGemmBlockK / 16; ++k) {
            umma_bf16(tmem_d, desc_advance(adesc, k * kAStep), desc_advance(bdesc, k * kBStep),
                      idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);  // smem slot reusable once these MMAs retire
          if (kb == kb1 - 1) umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue (warps 0-3) =====================
    int it = 0;
    uint32_t store_count = 0;   // staging-buffer parity of the TMA-store path
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int tmn = t % (num_n * num_m);
      const int n_blk = p.raster_m_fast ? tmn / num_m : tmn % num_n;
      const int m_blk = p.raster_m_fast ? tmn % num_m : tmn / num_n;
      const int split = t / (num_n * num_m);
      const int kb0 = split * kb_per_split;
      const bool has_k = kb0 < min(kb0 + kb_per_split, num_kb);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      if (!has_k) continue;  // (cannot happen: host clamps split_k) keeps roles in lock-step
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();

      const int row = m_blk * kGemmBlockM + warp * 32 + lane;
      const bool row_ok = row < p.M;
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + acc * BLOCK_N;
      const bf16* res_row = nullptr;
      if (p.residual != nullptr && row_ok) {
        const long long rr = p.res_row_mod > 0 ? (row % p.res_row_mod) : row;
        res_row = p.residual + rr * p.ldr;
      }
      if constexpr (EPI == EPI_STORE) {
        gemm_epilogue_store<BLOCK_N>(p, tmC, smem_c, taddr, warp, lane, m_blk, n_blk, split,
                                     store_count);
      } else if constexpr (EPI == EPI_NCE_FWD) {
        // Per row and column block: running maximum m and sum of 2^(x - m), x = s*log2(e), with an
        // online rescale per 32-column chunk (no fixed shift: a fixed exp(s - alpha) underflows
        // to sum = 0 once exp(temperature) reaches CLIP's usual logit scales of 50-100).
        const float alpha = __ldg(p.alpha_dev);
        const float a2 = alpha * 1.4426950408889634f;
        const int diag_col = row + p.diag_offset;
        float run_m = -INFINITY, run_s = 0.f;
#pragma unroll 1
        for (int c = 0; c < BLOCK_N / 32; ++c) {
          uint32_t v[32];
          tmem_ld_32x32(taddr + c * 32, v);
          tmem_ld_wait();
          const int col0 = n_blk * BLOCK_N + c * 32;
          if (col0 >= p.N) break;
          const bool interior = col0 + 32 <= p.N && (diag_col < col0 || diag_col >= col0 + 32);
          float cm = -INFINITY;
          if (interior) {
#pragma unroll
            for (int i = 0; i < 32; ++i) cm = fmaxf(cm, __uint_as_float(v[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int col = col0 + i;
              const bool is_diag = (col == diag_col);
              if (is_diag && row_ok) p.nce_pos[row] = __uint_as_float(v[i]) * alpha;
              if (col >= p.N || (p.dcl && is_diag)) v[i] = 0xff800000u;   // -inf: not in the sum
              cm = fmaxf(cm, __uint_as_float(v[i]));
            }
          }
          cm *= a2;                                   // a2 > 0: max commutes with the scaling
          if (cm > run_m) { run_s *= exp2f(run_m - cm); run_m = cm; }
          if (run_m > -INFINITY) {
#pragma unroll
            for (int i = 0; i < 32; ++i) run_s += exp2f(fmaf(__uint_as_float(v[i]), a2, -run_m));
          }
        }
        if (row_ok) {
          float2* dst = reinterpret_cast<float2*>(p.nce_part) + ((long long)n_blk * p.M + row);
          *dst = make_float2(run_m, run_s);
        }
      } else if constexpr (EPI == EPI_SEGMAX) {
        const float alpha = __ldg(p.alpha_dev);
        const int col_base = n_blk * n_stride;
        const int valid = min(n_stride, p.N - col_base);        // multiple of seg_len (and of 16)
        float best = -INFINITY;
        int best_i = 0;
#pragma unroll 1
        for (int c0 = 0; c0 < valid; c0 += 16) {
          uint32_t v[16];
          tmem_ld_32x16(taddr + c0, v);
          tmem_ld_wait();
          const int in_seg = c0 % p.seg_len;
          if (in_seg == 0) { best = -INFINITY; best_i = 0; }
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float sv = __uint_as_float(v[i]) * alpha;
            if (p.col_mul != nullptr)
              sv = fmaf(__uint_as_float(v[i]) * alpha, p.col_mul[col_base + c0 + i],
                        p.col_add[col_base + c0 + i]);
            if (sv > best) { best = sv; best_i = in_seg + i; }
          }
          if (in_seg + 16 == p.seg_len && row_ok) {
            const long long o = (long long)row * p.n_segs + (col_base + c0) / p.seg_len;
            p.seg_max[o] = best;
            p.seg_arg[o] = best_i;
          }
        }
      } else {
        const float alpha = __ldg(p.alpha_dev);
        const float gs = __ldg(p.gscale_dev);
        const float w_row = p.w_row * gs, w_col = p.w_col * gs, w_diag = p.w_diag * gs;
        const float a2 = alpha * 1.4426950408889634f;
        const int diag_col = row + p.diag_offset;
        const float lr2 = (row_ok && p.lse_row) ? p.lse_row[row] * 1.4426950408889634f : 0.f;
        float tsum = 0.f;
        // g leaves through swizzled 64-column boxes in shared memory and TMA stores (full 128-byte
        // lines; per-thread 16-byte row stores made this epilogue LSU-bound: 0.21 of the bf16 peak)
        const int row_in_tile = warp * 32 + lane;
#pragma unroll 1
        for (int q = 0; q < BLOCK_N / 64; ++q) {
          const uint32_t stg = smem_u32(smem_c) + (store_count & 1) * 16384;
          if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
          for (int c32 = 0; c32 < 2; ++c32) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + q * 64 + c32 * 32, v);
            tmem_ld_wait();
            const int col0 = n_blk * BLOCK_N + q * 64 + c32 * 32;
            float gq[32];
            // interior chunk (all 32 columns exist, the positive is elsewhere): ~10 instructions per
            // element, two ex2.approx each; the general path keeps the per-element predicates
            const bool interior = row_ok && col0 + 32 <= p.N && (diag_col < col0 || diag_col >= col0 + 32);
            if (interior) {
              float part = 0.f;
              if (p.w_col != 0.f) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  const float4 lc = __ldg(reinterpret_cast<const float4*>(p.lse_col + col0 + i));
                  const float l4[4] = {lc.x, lc.y, lc.z, lc.w};
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float acc_v = __uint_as_float(v[i + e]);
                    const float x = acc_v * a2;
                    float gv = w_col * nce_ex2(fmaf(l4[e], -1.4426950408889634f, x));
                    if (p.w_row != 0.f) gv = fmaf(w_row, nce_ex2(x - lr2), gv);
                    part = fmaf(gv, acc_v, part);
                    gq[i + e] = gv * alpha;
                  }
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const float acc_v = __uint_as_float(v[i]);
                  const float gv = w_row * nce_ex2(fmaf(acc_v, a2, -lr2));
                  part = fmaf(gv, acc_v, part);
                  gq[i] = gv * alpha;
                }
              }
              tsum = fmaf(part, alpha, tsum);
            } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int col = col0 + i;
              const float acc_v = __uint_as_float(v[i]);
              const bool is_diag = (col == diag_col);
              float gv = 0.f;
              if (row_ok && col < p.N) {
                if (!(p.dcl && is_diag)) {
                  if (p.w_row != 0.f) gv += w_row * nce_ex2(acc_v * a2 - lr2);
                  if (p.w_col != 0.f)
                    gv += w_col * nce_ex2(acc_v * a2 - __ldg(p.lse_col + col) * 1.4426950408889634f);
                }
                if (is_diag) gv -= w_diag;
                tsum += gv * acc_v * alpha;
              }
              gq[i] = gv * alpha;   // temperature folded in: d rows = gq @ cols; 0 beyond N / M
            }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(
                               stg + swz128(row_in_tile, c32 * 4 + i)),
                           "r"(pack_bf16x2(gq[i * 8 + 0], gq[i * 8 + 1])),
                           "r"(pack_bf16x2(gq[i * 8 + 2], gq[i * 8 + 3])),
                           "r"(pack_bf16x2(gq[i * 8 + 4], gq[i * 8 + 5])),
                           "r"(pack_bf16x2(gq[i * 8 + 6], gq[i * 8 + 7]))
                           : "memory");
            }
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (threadIdx.x == 0) {
            const int c0 = n_blk * BLOCK_N + q * 64;
            if (c0 < (int)p.ldc) {      // the map spans ldc = roundup8(N) columns: the pad columns get zeros
              asm volatile(
                  "cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                      reinterpret_cast<uint64_t>(&tmC)),
                  "r"(stg), "r"(c0), "r"(m_blk * kGemmBlockM)
                  : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          ++store_count;
        }
        if (p.dtemp != nullptr) {
          tsum = warp_sum(tsum);
          if (lane == 0) atomicAdd(p.dtemp, tsum);
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
    if (((EPI == EPI_STORE && p.use_tma_store) || EPI == EPI_NCE_BWD) && threadIdx.x == 0)
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 5) {
    tcgen05_fence_after();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

}  // namespace xclip
