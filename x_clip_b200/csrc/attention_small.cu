// Fused multi-head attention for SHORT sequences (n <= 128, dim_head = 64), sm_100a tcgen05.
//
// Same math as attention_fwd.cu / attention_bwd.cu (reference x_clip/x_clip.py:217-244 and its
// autograd backward) but organised for many small (batch, head) items - the ViT-B/16 tower with
// patch dropout (n = 98), the 77-token text tower (n = 78) and the README image tower (n = 32):
// one item is a single 128-row tile whose latency chain (TMA -> S MMA -> softmax -> PV MMA ->
// store) cannot be hidden inside one CTA, so the kernels are small enough that SEVERAL CTAs are
// resident per SM and the hardware overlaps the phases of different items.
//
//   forward : ROWS = 128 -> 5 warps (4 softmax, 1 control), 49 KiB smem, 128 TMEM columns,
//             4 CTAs / SM;  ROWS = 64 (n <= 64) -> 3 warps, 25 KiB, 64 columns, 8 CTAs / SM.
//             A query row is owned by ONE thread (tcgen05.ld 32x32b hands a lane its whole row),
//             so the row max / sum need no cross-thread exchange.  P (bf16) overwrites the dead
//             Q|K buffers, O overwrites the dead S columns.
//   backward: 9 warps (8 compute: two threads per query row, half the keys each; no reductions
//             are needed because lse and delta are inputs), operands sized by ceil16(n), dV/dK/dQ
//             accumulators overwrite the dead S/dP columns (256 TMEM columns), 2 CTAs / SM for
//             n <= 112.
//
// Masking semantics are the reference's: masked keys get -FLT_MAX AFTER scaling (a fully masked
// row attends uniformly), keys >= n do not exist; `causal` additionally masks keys j > i
// (x_clip.py:233-236).  Items without any masked key take a table-free fast path.
#include "common.cuh"
#include "host.h"

namespace xclip {

constexpr int kSDh = 64;

struct AttnSmallFwdParams {
  int B, H, n, nkp;        // nkp = ceil16(n)
  float scale_log2;        // dim_head^-0.5 * log2(e)  (> 0)
  const uint8_t* mask;     // [B, n] (1 = attend) or null
  bf16* o;
  long long ldo;
  float* lse;              // [B, H, n] base-2 log-sum-exp of the scaled, masked scores
};

__device__ __forceinline__ float sm_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void sm_sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                          uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c),
               "r"(d)
               : "memory");
}
__device__ __forceinline__ float4 sm_lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "r"(addr));
  return v;
}
__device__ __forceinline__ void sm_sts_f(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ uint32_t sm_lds_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sm_sts_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

template <uint32_t kCols>
__device__ __forceinline__ void sm_tmem_alloc(uint32_t* smem_result) {
  static_assert(kCols == 64 || kCols == 128 || kCols == 256, "");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_result)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}

// One 32- or 16-column chunk of a row: raw scores -> t (scaled, masked, base-2 domain).
//   fast path : no masked key in this item and no causal mask: t = raw * c, columns >= valid are
//               -inf (they only occur in the last chunk).
//   table path: t = fma(raw, mul[j], add[j]) (mul = c or 0, add = 0 / -FLT_MAX / -inf).
template <int CNT, bool kCausal>
__device__ __forceinline__ void sm_scores(const uint32_t (&v)[32], float (&t)[32], bool fast,
                                          int valid, float c, uint32_t mul_addr, uint32_t add_addr,
                                          int col0, int row) {
  if (fast) {
    if (valid >= CNT) {
#pragma unroll
      for (int i = 0; i < CNT; ++i) t[i] = __uint_as_float(v[i]) * c;
    } else {
#pragma unroll
      for (int i = 0; i < CNT; ++i) t[i] = i < valid ? __uint_as_float(v[i]) * c : -INFINITY;
    }
  } else {
#pragma unroll
    for (int i = 0; i < CNT; i += 4) {
      const float4 m = sm_lds_f4(mul_addr + i * 4);
      const float4 a = sm_lds_f4(add_addr + i * 4);
      t[i] = fmaf(__uint_as_float(v[i]), m.x, a.x);
      t[i + 1] = fmaf(__uint_as_float(v[i + 1]), m.y, a.y);
      t[i + 2] = fmaf(__uint_as_float(v[i + 2]), m.z, a.z);
      t[i + 3] = fmaf(__uint_as_float(v[i + 3]), m.w, a.w);
    }
    if constexpr (kCausal) {
#pragma unroll
      for (int i = 0; i < CNT; ++i)
        if (col0 + i > row) t[i] = fminf(t[i], -FLT_MAX);   // (-inf of a non-existent key stays)
    }
  }
}

template <int ROWS, bool kCausal>
__global__ void __launch_bounds__((ROWS / 32 + 1) * 32, ROWS == 128 ? 4 : 8)
attn_fwd_small_kernel(const __grid_constant__ CUtensorMap tm_qkv, const AttnSmallFwdParams p) {
  constexpr int NSW = ROWS / 32;                 // softmax warps; warp NSW is the control warp
  constexpr int kBox = ROWS * 128;               // bytes of one [ROWS x 64] bf16 TMA box
  constexpr int kPBlk = 128 * 128;               // one [128 rows x 64 keys] bf16 block of P
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sQ = smem;                            // Q | K, later overwritten by P
  uint8_t* sK = sQ + kBox;
  uint8_t* sV = sK + kBox;
  uint8_t* tail = sV + kBox;
  uint64_t* qk_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* v_bar = qk_bar + 1;
  uint64_t* s_bar = qk_bar + 2;
  uint64_t* p_bar = qk_bar + 3;
  uint64_t* o_bar = qk_bar + 4;
  uint64_t* e_bar = qk_bar + 5;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(qk_bar + 6);
  const uint32_t sFlag = smem_u32(tail + 64);            // [2][4] u32: "this warp saw a masked key"
  const uint32_t sMul = smem_u32(tail + 128);            // [2][ROWS] f32
  const uint32_t sAdd = sMul + 2 * ROWS * 4;             // [2][ROWS] f32

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool is_control = warp == NSW;

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    mbar_init(qk_bar, 1);
    mbar_init(v_bar, 1);
    mbar_init(s_bar, 1);
    mbar_init(p_bar, NSW);
    mbar_init(o_bar, 1);
    mbar_init(e_bar, NSW);
    fence_barrier_init();
  }
  if (is_control) {
    if (lane == 0) tma_prefetch_desc(&tm_qkv);
    sm_tmem_alloc<ROWS>(tmem_slot);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int inner = p.H * kSDh;
  const int total = p.B * p.H;

  if (is_control) {
    if (XCLIP_ONE_LANE(lane)) {
      const uint64_t desc_q = make_smem_desc(smem_u32(sQ), 0, 1024);
      const uint64_t desc_k = make_smem_desc(smem_u32(sK), 0, 1024);
      const uint64_t desc_p = make_smem_desc(smem_u32(sQ), 0, 1024);
      const uint64_t desc_v = make_smem_desc(smem_u32(sV), 8192, 1024);
      const uint32_t idesc_s = make_idesc_bf16(128, p.nkp, kMajorK, kMajorK);
      constexpr uint32_t idesc_pv = make_idesc_bf16(128, kSDh, kMajorK, kMajorMN);
      const int ksteps = p.nkp / 16;
      uint32_t it = 0;
      for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++it) {
        const int b = bh / p.H, h = bh - b * p.H;
        const uint32_t par = it & 1;
        // (the previous item's PV retired - waited below - so Q|K/P and V smem are free)
        mbar_arrive_expect_tx(qk_bar, 2 * kBox);
        tma_load_3d(sQ, &tm_qkv, qk_bar, h * kSDh, 0, b);
        tma_load_3d(sK, &tm_qkv, qk_bar, inner + h * kSDh, 0, b);
        mbar_arrive_expect_tx(v_bar, kBox);
        tma_load_3d(sV, &tm_qkv, v_bar, 2 * inner + h * kSDh, 0, b);
        if (it > 0) mbar_wait(e_bar, par ^ 1);   // O of the previous item was read out of TMEM
        mbar_wait(qk_bar, par);
        tcgen05_fence_after();
#pragma unroll
        for (int k = 0; k < kSDh / 16; ++k)
          umma_bf16(tmem_base, desc_q + 2 * k, desc_k + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        umma_commit(s_bar);
        mbar_wait(p_bar, par);                   // P in smem, S consumed
        mbar_wait(v_bar, par);
        tcgen05_fence_after();
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          if (k < ksteps)
            umma_bf16(tmem_base, desc_p + ((k >> 2) * (kPBlk >> 4) + (k & 3) * 2), desc_v + k * 128,
                      idesc_pv, k > 0 ? 1u : 0u);
        }
        umma_commit(o_bar);
        mbar_wait(o_bar, par);
      }
    }
    __syncwarp();
  } else {
    const int row = warp * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);
    const bool alive = warp * 32 < p.n;
    const float c = p.scale_log2;
    uint32_t it = 0;
    // the key-mask byte of the CTA's NEXT item is fetched while the current one is computed
    bool keep_n = true;
    auto fetch_mask = [&](int bh2) {
      keep_n = true;
      if (p.mask != nullptr && bh2 < total && (int)threadIdx.x < p.n)
        keep_n = __ldg(p.mask + (long long)(bh2 / p.H) * p.n + threadIdx.x) != 0;
    };
    fetch_mask(blockIdx.x);
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++it) {
      const int b = bh / p.H, h = bh - b * p.H;
      const uint32_t par = it & 1;
      // ---- per-key tables (double buffered by item parity) + "any key masked" flag
      {
        const int j = threadIdx.x;               // 0 .. ROWS-1
        float mul = 0.f, add = -INFINITY;
        bool masked = false;
        if (j < p.n) {
          const bool keep = keep_n;
          mul = keep ? c : 0.f;
          add = keep ? 0.f : -FLT_MAX;
          masked = !keep;
        }
        fetch_mask(bh + (int)gridDim.x);
        sm_sts_f(sMul + (par * ROWS + j) * 4, mul);
        sm_sts_f(sAdd + (par * ROWS + j) * 4, add);
        const uint32_t any = __ballot_sync(0xffffffffu, masked);
        if (lane == 0) sm_sts_u32(sFlag + (par * 4 + warp) * 4, any);
      }
      asm volatile("bar.sync 1, %0;" ::"n"(NSW * 32) : "memory");
      uint32_t anym = 0;
#pragma unroll
      for (int w = 0; w < NSW; ++w) anym |= sm_lds_u32(sFlag + (par * 4 + w) * 4);
      const bool fast = !kCausal && anym == 0;
      const uint32_t mulb = sMul + par * ROWS * 4, addb = sAdd + par * ROWS * 4;

      mbar_wait(s_bar, par);
      tcgen05_fence_after();
      float m2 = -INFINITY, sum = 0.f;
      if (alive && fast) {
        // ---- table-free path (no masked key, not causal): the scale is positive, so the row maximum is
        // taken over the RAW scores (one FMNMX per element) and scaled once; pass 2 is one FFMA + one
        // MUFU.EX2 per element:  p = 2^(raw * c - m2)
        float mr = -INFINITY;
        for (int c0 = 0; c0 < p.nkp; c0 += 16) {         // (16-column steps: nkp is a multiple of 16)
          const int valid = p.n - c0;
          uint32_t w[16];
          tmem_ld_32x16(t_row + c0, w);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (valid >= 16 || i < valid) mr = fmaxf(mr, __uint_as_float(w[i]));
        }
        m2 = mr * c;
        const float nm2 = -m2;
        for (int c0 = 0; c0 < p.nkp; c0 += 16) {
          const int valid = p.n - c0;
          uint32_t w[16];
          tmem_ld_32x16(t_row + c0, w);
          tmem_ld_wait();
          const uint32_t blk = smem_u32(sQ) + (c0 >> 6) * kPBlk;
          const int chunk0 = (c0 & 63) >> 3;
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
            float e[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float x = sm_ex2(fmaf(__uint_as_float(w[cc * 8 + i]), c, nm2));
              e[i] = (valid >= 16 || cc * 8 + i < valid) ? x : 0.f;
            }
            sum += ((e[0] + e[1]) + (e[2] + e[3])) + ((e[4] + e[5]) + (e[6] + e[7]));
            sm_sts_v4(blk + swz128(row, chunk0 + cc), pack_bf16x2(e[0], e[1]),
                      pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
          }
        }
      } else if (alive) {
        // ---- pass 1: row maximum
        for (int c0 = 0; c0 < p.nkp; c0 += 32) {
          uint32_t v[32];
          float t[32];
          if (p.nkp - c0 >= 32) {
            tmem_ld_32x32(t_row + c0, v);
            tmem_ld_wait();
            sm_scores<32, kCausal>(v, t, fast, p.n - c0, c, mulb + c0 * 4, addb + c0 * 4, c0, row);
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              m2 = fmaxf(m2, fmaxf(fmaxf(t[i], t[i + 1]), fmaxf(t[i + 2], t[i + 3])));
          } else {
            uint32_t w[16];
            tmem_ld_32x16(t_row + c0, w);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = w[i];
            sm_scores<16, kCausal>(v, t, fast, p.n - c0, c, mulb + c0 * 4, addb + c0 * 4, c0, row);
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              m2 = fmaxf(m2, fmaxf(fmaxf(t[i], t[i + 1]), fmaxf(t[i + 2], t[i + 3])));
          }
        }
        // ---- pass 2: probabilities -> bf16 P (SW128 K-major blocks of 64 keys), row sum
        for (int c0 = 0; c0 < p.nkp; c0 += 32) {
          uint32_t v[32];
          float t[32];
          const bool full = p.nkp - c0 >= 32;
          if (full) {
            tmem_ld_32x32(t_row + c0, v);
            tmem_ld_wait();
            sm_scores<32, kCausal>(v, t, fast, p.n - c0, c, mulb + c0 * 4, addb + c0 * 4, c0, row);
          } else {
            uint32_t w[16];
            tmem_ld_32x16(t_row + c0, w);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = w[i];
            sm_scores<16, kCausal>(v, t, fast, p.n - c0, c, mulb + c0 * 4, addb + c0 * 4, c0, row);
          }
          const uint32_t blk = smem_u32(sQ) + (c0 >> 6) * kPBlk;
          const int chunk0 = (c0 & 63) >> 3;
#pragma unroll
          for (int cc = 0; cc < 4; ++cc) {
            if (cc < 2 || full) {
              float e[8];
#pragma unroll
              for (int i = 0; i < 8; ++i) e[i] = sm_ex2(t[cc * 8 + i] - m2);
              sum += ((e[0] + e[1]) + (e[2] + e[3])) + ((e[4] + e[5]) + (e[6] + e[7]));
              sm_sts_v4(blk + swz128(row, chunk0 + cc), pack_bf16x2(e[0], e[1]),
                        pack_bf16x2(e[2], e[3]), pack_bf16x2(e[4], e[5]), pack_bf16x2(e[6], e[7]));
            }
          }
        }
      }
      fence_proxy_async_smem();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_bar);

      // ---- epilogue: O / sum -> bf16, log-sum-exp
      mbar_wait(o_bar, par);
      tcgen05_fence_after();
      if (alive) {
        const float inv = 1.f / sum;
        uint32_t v0[32], v1[32];
        tmem_ld_32x32(t_row, v0);
        tmem_ld_32x32(t_row + 32, v1);
        tmem_ld_wait();
        if (row < p.n) {
          p.lse[((long long)b * p.H + h) * p.n + row] = m2 + log2f(sum);
          bf16* dst = p.o + ((long long)b * p.n + row) * p.ldo + h * kSDh;
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(v0[i]) * inv, __uint_as_float(v0[i + 1]) * inv);
            o.y = pack_bf16x2(__uint_as_float(v0[i + 2]) * inv, __uint_as_float(v0[i + 3]) * inv);
            o.z = pack_bf16x2(__uint_as_float(v0[i + 4]) * inv, __uint_as_float(v0[i + 5]) * inv);
            o.w = pack_bf16x2(__uint_as_float(v0[i + 6]) * inv, __uint_as_float(v0[i + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + i) = o;
          }
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(v1[i]) * inv, __uint_as_float(v1[i + 1]) * inv);
            o.y = pack_bf16x2(__uint_as_float(v1[i + 2]) * inv, __uint_as_float(v1[i + 3]) * inv);
            o.z = pack_bf16x2(__uint_as_float(v1[i + 4]) * inv, __uint_as_float(v1[i + 5]) * inv);
            o.w = pack_bf16x2(__uint_as_float(v1[i + 6]) * inv, __uint_as_float(v1[i + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + 32 + i) = o;
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(e_bar);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (is_control) {
    tcgen05_fence_after();
    tmem_dealloc<ROWS>(tmem_base);
  }
}

template <int ROWS, bool kCausal>
static int launch_fwd_small(const void* qkv, int64_t ld_qkv, const AttnSmallFwdParams& p,
                            cudaStream_t stream) {
  constexpr int kThreads = (ROWS / 32 + 1) * 32;
  constexpr int kSmem = 3 * ROWS * 128 + 128 + 4 * ROWS * 4;
  constexpr int kPerSm = ROWS == 128 ? 4 : 8;
  CUtensorMap tm;
  int rc = encode_3d_bf16(&tm, qkv, (uint64_t)(3 * p.H * kSDh), (uint64_t)p.n, (uint64_t)p.B,
                          (uint64_t)ld_qkv, (uint64_t)p.n * ld_qkv, kSDh, ROWS);
  if (rc) return rc;
  auto kern = attn_fwd_small_kernel<ROWS, kCausal>;
  rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), kSmem);
  if (rc) return rc;
  long long grid = (long long)num_sms() * kPerSm;
  if (grid > (long long)p.B * p.H) grid = (long long)p.B * p.H;
  kern<<<(int)grid, kThreads, kSmem, stream>>>(tm, p);
  XCLIP_LAUNCH_CHECK("attn_fwd_small_kernel");
  return XCLIP_OK;
}

// =============================================================================================
// backward
// =============================================================================================
struct AttnSmallBwdParams {
  int B, H, n, nkp;
  float scale, scale_log2;
  const uint8_t* mask;   // [B, n] or null
  const float* lse;      // [B, H, n] base-2
  const float* delta;    // [B, H, n] rowsum(dO * O)
  bf16* dqkv;            // [B*n, ld]: dq | dk | dv
  long long ld;
};

constexpr int kSBwdComputeWarps = 8;
constexpr int kSBwdThreads = (kSBwdComputeWarps + 1) * 32;

// smem: Q | K | dO | P block 0 (= V until S/dP retired) | P block 1 | dS block 0 | dS block 1, every
// buffer nkp*128 bytes ("box"); K-major A reads of Q / dO / dS touch 128 rows (16 KiB) from a
// buffer's base, so the allocation extends 16 KiB past the start of the last dS block.
__host__ __device__ constexpr int sbwd_smem_bytes(int nkp) {
  const int box = nkp * 128;
  const int body = (7 * box > 6 * box + 16384) ? 7 * box : 6 * box + 16384;
  return body + 128 + 4 * 128 * 4 + 64;
}

template <bool kCausal>
__global__ void __launch_bounds__(kSBwdThreads, 2)
attn_bwd_small_kernel(const __grid_constant__ CUtensorMap tm_qkv,
                      const __grid_constant__ CUtensorMap tm_do, const AttnSmallBwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int box = p.nkp * 128;
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + box;
  uint8_t* sdO = sK + box;
  uint8_t* sP = sdO + box;            // block 0 doubles as the V buffer
  uint8_t* sdS = sP + 2 * box;
  const int body = (7 * box > 6 * box + 16384) ? 7 * box : 6 * box + 16384;
  uint8_t* tail = smem + body;
  uint64_t* qk_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* vdo_bar = qk_bar + 1;
  uint64_t* s_bar = qk_bar + 2;
  uint64_t* pds_bar = qk_bar + 3;
  uint64_t* dq_bar = qk_bar + 4;
  uint64_t* g_bar = qk_bar + 5;
  uint64_t* e_bar = qk_bar + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(qk_bar + 7);
  const uint32_t sFlag = smem_u32(tail + 64);           // [2][4] u32
  const uint32_t sMul = smem_u32(tail + 128);           // [2][128] f32
  const uint32_t sAdd = sMul + 2 * 128 * 4;             // [2][128] f32

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const bool is_control = warp == kSBwdComputeWarps;

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    mbar_init(qk_bar, 1);
    mbar_init(vdo_bar, 1);
    mbar_init(s_bar, 1);
    mbar_init(pds_bar, kSBwdComputeWarps);
    mbar_init(dq_bar, 1);
    mbar_init(g_bar, 1);
    mbar_init(e_bar, kSBwdComputeWarps);
    fence_barrier_init();
  }
  if (is_control) {
    if (lane == 0) {
      tma_prefetch_desc(&tm_qkv);
      tma_prefetch_desc(&tm_do);
    }
    sm_tmem_alloc<256>(tmem_slot);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // S [0,128), dP [128,256); once P/dS are in smem: dV [0,64), dK [64,128), dQ [128,192)
  const uint32_t tS = tmem_base, tdP = tmem_base + 128, tdV = tmem_base, tdK = tmem_base + 64,
                 tdQ = tmem_base + 128;
  const int inner = p.H * kSDh;
  const int total = p.B * p.H;

  if (is_control) {
    if (XCLIP_ONE_LANE(lane)) {
      const uint32_t idesc_s = make_idesc_bf16(128, p.nkp, kMajorK, kMajorK);
      constexpr uint32_t idesc_t = make_idesc_bf16(128, kSDh, kMajorMN, kMajorMN);
      constexpr uint32_t idesc_q = make_idesc_bf16(128, kSDh, kMajorK, kMajorMN);
      const uint64_t desc_q = make_smem_desc(smem_u32(sQ), 0, 1024);
      const uint64_t desc_k = make_smem_desc(smem_u32(sK), 0, 1024);
      const uint64_t desc_do = make_smem_desc(smem_u32(sdO), 0, 1024);
      const uint64_t desc_v = make_smem_desc(smem_u32(sP), 0, 1024);
      const uint64_t desc_pT = make_smem_desc(smem_u32(sP), box, 1024);     // MN-major A
      const uint64_t desc_dsT = make_smem_desc(smem_u32(sdS), box, 1024);   // MN-major A
      const uint64_t desc_dsK = make_smem_desc(smem_u32(sdS), 0, 1024);     // K-major A
      const uint64_t desc_kmn = make_smem_desc(smem_u32(sK), 8192, 1024);   // MN-major B
      const uint64_t desc_qmn = make_smem_desc(smem_u32(sQ), 8192, 1024);
      const uint64_t desc_domn = make_smem_desc(smem_u32(sdO), 8192, 1024);
      const int ksteps = p.nkp / 16;
      const uint32_t blk16 = static_cast<uint32_t>(box) >> 4;
      uint32_t it = 0;
      for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++it) {
        const int b = bh / p.H, h = bh - b * p.H;
        const uint32_t par = it & 1;
        // (all MMAs of the previous item retired - g_bar was waited for below)
        mbar_arrive_expect_tx(qk_bar, 2 * box);
        tma_load_3d(sQ, &tm_qkv, qk_bar, h * kSDh, 0, b);
        tma_load_3d(sK, &tm_qkv, qk_bar, inner + h * kSDh, 0, b);
        mbar_arrive_expect_tx(vdo_bar, 2 * box);
        tma_load_3d(sP, &tm_qkv, vdo_bar, 2 * inner + h * kSDh, 0, b);
        tma_load_3d(sdO, &tm_do, vdo_bar, h * kSDh, 0, b);
        if (it > 0) mbar_wait(e_bar, par ^ 1);   // dQ/dK/dV of the previous item left TMEM
        mbar_wait(qk_bar, par);
        tcgen05_fence_after();
#pragma unroll
        for (int k = 0; k < kSDh / 16; ++k)
          umma_bf16(tS, desc_q + 2 * k, desc_k + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        mbar_wait(vdo_bar, par);
        tcgen05_fence_after();
#pragma unroll
        for (int k = 0; k < kSDh / 16; ++k)
          umma_bf16(tdP, desc_do + 2 * k, desc_v + 2 * k, idesc_s, k > 0 ? 1u : 0u);
        umma_commit(s_bar);
        mbar_wait(pds_bar, par);                 // P, dS in smem; S/dP columns consumed
        tcgen05_fence_after();
#pragma unroll
        for (int k = 0; k < 8; ++k) {            // dQ = dS K   (contraction over keys)
          if (k < ksteps)
            umma_bf16(tdQ, desc_dsK + ((k >> 2) * blk16 + (k & 3) * 2), desc_kmn + k * 128, idesc_q,
                      k > 0 ? 1u : 0u);
        }
        umma_commit(dq_bar);
#pragma unroll
        for (int k = 0; k < 8; ++k) {            // dV = P^T dO, dK = dS^T Q (contraction over queries)
          if (k < ksteps) {
            umma_bf16(tdV, desc_pT + k * 128, desc_domn + k * 128, idesc_t, k > 0 ? 1u : 0u);
            umma_bf16(tdK, desc_dsT + k * 128, desc_qmn + k * 128, idesc_t, k > 0 ? 1u : 0u);
          }
        }
        umma_commit(g_bar);
        mbar_wait(g_bar, par);
      }
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3, half = warp >> 2;
    const int row = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const bool alive = quarter * 32 < p.nkp;
    const int nch = p.nkp / 16;
    const int cb = half == 0 ? 0 : (nch + 1) / 2;
    const int ce = half == 0 ? (nch + 1) / 2 : nch;
    const float c = p.scale_log2;
    uint32_t it = 0;
    // per-row scalars (and the key-mask byte) of the CTA's NEXT item are fetched while the current one
    // is computed: their global-load latency was the top stall of this kernel (ncu: 33 % L1TEX scoreboard)
    float lse_n = INFINITY, delta_n = 0.f;      // +inf log-sum-exp -> p = 0 for the padding rows [n, nkp)
    bool keep_n = false;
    auto fetch = [&](int bh2) {
      lse_n = INFINITY; delta_n = 0.f; keep_n = false;
      if (bh2 < total) {
        const int b2 = bh2 / p.H;
        if (row < p.n) {
          lse_n = __ldg(p.lse + (long long)bh2 * p.n + row);
          delta_n = __ldg(p.delta + (long long)bh2 * p.n + row);
        }
        if (threadIdx.x < 128 && threadIdx.x < p.n)
          keep_n = p.mask ? (__ldg(p.mask + (long long)b2 * p.n + threadIdx.x) != 0) : true;
      }
    };
    fetch(blockIdx.x);
    for (int bh = blockIdx.x; bh < total; bh += gridDim.x, ++it) {
      const int b = bh / p.H, h = bh - b * p.H;
      const uint32_t par = it & 1;
      const float lse_i = lse_n, delta_i = delta_n;
      if (threadIdx.x < 128) {
        const int j = threadIdx.x;
        const bool keep = keep_n;                // (false for j >= n)
        sm_sts_f(sMul + (par * 128 + j) * 4, keep ? c : 0.f);
        sm_sts_f(sAdd + (par * 128 + j) * 4, keep ? 0.f : -INFINITY);
        const uint32_t any = __ballot_sync(0xffffffffu, j < p.n && !keep);
        if (lane == 0) sm_sts_u32(sFlag + (par * 4 + warp) * 4, any);
      }
      fetch(bh + (int)gridDim.x);
      const float dsc = delta_i * p.scale;
      asm volatile("bar.sync 1, 256;" ::: "memory");
      uint32_t anym = 0;
#pragma unroll
      for (int w = 0; w < 4; ++w) anym |= sm_lds_u32(sFlag + (par * 4 + w) * 4);
      const bool fast = !kCausal && anym == 0;
      const uint32_t mulb = sMul + par * 128 * 4, addb = sAdd + par * 128 * 4;

      mbar_wait(s_bar, par);
      tcgen05_fence_after();
      if (alive) {
        for (int ch = cb; ch < ce; ++ch) {
          const int c0 = ch * 16;
          uint32_t sv[16], dv[16];
          tmem_ld_32x16(tS + lane_off + c0, sv);
          tmem_ld_32x16(tdP + lane_off + c0, dv);
          tmem_ld_wait();
          float pr[16], ds[16];
          if (fast && p.n - c0 >= 16) {
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const float pv = sm_ex2(fmaf(__uint_as_float(sv[e]), c, -lse_i));
              pr[e] = pv;
              ds[e] = pv * fmaf(__uint_as_float(dv[e]), p.scale, -dsc);
            }
          } else {
#pragma unroll
            for (int e = 0; e < 16; e += 4) {
              const float4 m = sm_lds_f4(mulb + (c0 + e) * 4);
              const float4 a = sm_lds_f4(addb + (c0 + e) * 4);
              const float mm[4] = {m.x, m.y, m.z, m.w}, aa[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                float t = fmaf(__uint_as_float(sv[e + u]), mm[u], aa[u]);
                if (kCausal && c0 + e + u > row) t = -INFINITY;
                const float pv = sm_ex2(t - lse_i);
                pr[e + u] = pv;
                ds[e + u] = pv * fmaf(__uint_as_float(dv[e + u]), p.scale, -dsc);
              }
            }
          }
          if (row < p.nkp) {
            const uint32_t pblk = smem_u32(sP) + (c0 >> 6) * box;
            const uint32_t dblk = smem_u32(sdS) + (c0 >> 6) * box;
            const int chunk0 = (c0 & 63) >> 3;
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
              sm_sts_v4(pblk + swz128(row, chunk0 + cc), pack_bf16x2(pr[cc * 8 + 0], pr[cc * 8 + 1]),
                        pack_bf16x2(pr[cc * 8 + 2], pr[cc * 8 + 3]),
                        pack_bf16x2(pr[cc * 8 + 4], pr[cc * 8 + 5]),
                        pack_bf16x2(pr[cc * 8 + 6], pr[cc * 8 + 7]));
              sm_sts_v4(dblk + swz128(row, chunk0 + cc), pack_bf16x2(ds[cc * 8 + 0], ds[cc * 8 + 1]),
                        pack_bf16x2(ds[cc * 8 + 2], ds[cc * 8 + 3]),
                        pack_bf16x2(ds[cc * 8 + 4], ds[cc * 8 + 5]),
                        pack_bf16x2(ds[cc * 8 + 6], ds[cc * 8 + 7]));
            }
          }
        }
      }
      fence_proxy_async_smem();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(pds_bar);

      // dQ: this thread converts 32 of the 64 columns of its query row
      mbar_wait(dq_bar, par);
      tcgen05_fence_after();
      if (alive) {
        uint32_t v[32];
        tmem_ld_32x32(tdQ + lane_off + half * 32, v);
        tmem_ld_wait();
        if (row < p.n) {
          bf16* dst = p.dqkv + ((long long)b * p.n + row) * p.ld + h * kSDh + half * 32;
#pragma unroll
          for (int e = 0; e < 32; e += 8) {
            uint4 o;
            o.x = pack_bf16x2(__uint_as_float(v[e]), __uint_as_float(v[e + 1]));
            o.y = pack_bf16x2(__uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]));
            o.z = pack_bf16x2(__uint_as_float(v[e + 4]), __uint_as_float(v[e + 5]));
            o.w = pack_bf16x2(__uint_as_float(v[e + 6]), __uint_as_float(v[e + 7]));
            *reinterpret_cast<uint4*>(dst + e) = o;
          }
        }
      }
      // dK (half 0) / dV (half 1): the thread's row is a KEY index here
      mbar_wait(g_bar, par);
      tcgen05_fence_after();
      if (alive) {
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          uint32_t v[32];
          tmem_ld_32x32((half == 0 ? tdK : tdV) + lane_off + cc * 32, v);
          tmem_ld_wait();
          if (row < p.n) {
            bf16* dst = p.dqkv + ((long long)b * p.n + row) * p.ld + (half + 1) * inner + h * kSDh +
                        cc * 32;
#pragma unroll
            for (int e = 0; e < 32; e += 8) {
              uint4 o;
              o.x = pack_bf16x2(__uint_as_float(v[e]), __uint_as_float(v[e + 1]));
              o.y = pack_bf16x2(__uint_as_float(v[e + 2]), __uint_as_float(v[e + 3]));
              o.z = pack_bf16x2(__uint_as_float(v[e + 4]), __uint_as_float(v[e + 5]));
              o.w = pack_bf16x2(__uint_as_float(v[e + 6]), __uint_as_float(v[e + 7]));
              *reinterpret_cast<uint4*>(dst + e) = o;
            }
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(e_bar);
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (is_control) {
    tcgen05_fence_after();
    tmem_dealloc<256>(tmem_base);
  }
}

// host entry used by xclip_attn_bwd (attention_bwd.cu) for n <= 128; delta is already computed
int attn_bwd_small(const void* qkv, int64_t ld_qkv, const uint8_t* key_mask, const void* d_o,
                   int64_t lddo, const float* lse, const float* delta, void* dqkv, int64_t ld_dqkv,
                   int B, int n, int heads, float scale, int causal, cudaStream_t stream) {
  XCLIP_REQUIRE(n <= 128, "attn_bwd_small: n=%d > 128", n);
  XCLIP_REQUIRE(scale > 0.f, "attn_bwd_small: scale must be positive");
  AttnSmallBwdParams p;
  p.B = B; p.H = heads; p.n = n; p.nkp = (n + 15) / 16 * 16;
  p.scale = scale; p.scale_log2 = scale * 1.4426950408889634f;
  p.mask = key_mask; p.lse = lse; p.delta = delta;
  p.dqkv = reinterpret_cast<bf16*>(dqkv); p.ld = ld_dqkv;
  CUtensorMap tq, tdo;
  int rc = encode_3d_bf16(&tq, qkv, (uint64_t)(3 * heads * kSDh), (uint64_t)n, (uint64_t)B,
                          (uint64_t)ld_qkv, (uint64_t)n * ld_qkv, kSDh, (uint32_t)p.nkp);
  if (rc) return rc;
  rc = encode_3d_bf16(&tdo, d_o, (uint64_t)(heads * kSDh), (uint64_t)n, (uint64_t)B, (uint64_t)lddo,
                      (uint64_t)n * lddo, kSDh, (uint32_t)p.nkp);
  if (rc) return rc;
  const int smem = sbwd_smem_bytes(p.nkp);
  rc = ensure_dynamic_smem(causal ? reinterpret_cast<const void*>(attn_bwd_small_kernel<true>)
                                  : reinterpret_cast<const void*>(attn_bwd_small_kernel<false>),
                           sbwd_smem_bytes(128));
  if (rc) return rc;
  int per_sm = (227 * 1024) / (smem + 1024);
  if (per_sm > 2) per_sm = 2;      // 256 TMEM columns per CTA
  if (per_sm < 1) per_sm = 1;
  long long grid = (long long)num_sms() * per_sm;
  if (grid > (long long)B * heads) grid = (long long)B * heads;
  if (causal)
    attn_bwd_small_kernel<true><<<(int)grid, kSBwdThreads, smem, stream>>>(tq, tdo, p);
  else
    attn_bwd_small_kernel<false><<<(int)grid, kSBwdThreads, smem, stream>>>(tq, tdo, p);
  XCLIP_LAUNCH_CHECK("attn_bwd_small_kernel");
  return XCLIP_OK;
}

// host entry used by xclip_attn_fwd (attention_fwd.cu) for n <= 128
int attn_fwd_small(const void* qkv, int64_t ld_qkv, const uint8_t* key_mask, void* o, int64_t ldo,
                   float* lse, int B, int n, int heads, float scale, int causal,
                   cudaStream_t stream) {
  XCLIP_REQUIRE(n <= 128, "attn_fwd_small: n=%d > 128", n);
  XCLIP_REQUIRE(scale > 0.f, "attn_fwd_small: scale must be positive");
  AttnSmallFwdParams p;
  p.B = B; p.H = heads; p.n = n; p.nkp = (n + 15) / 16 * 16;
  p.scale_log2 = scale * 1.4426950408889634f;
  p.mask = key_mask;
  p.o = reinterpret_cast<bf16*>(o);
  p.ldo = ldo;
  p.lse = lse;
  if (n <= 64)
    return causal ? launch_fwd_small<64, true>(qkv, ld_qkv, p, stream)
                  : launch_fwd_small<64, false>(qkv, ld_qkv, p, stream);
  return causal ? launch_fwd_small<128, true>(qkv, ld_qkv, p, stream)
                : launch_fwd_small<128, false>(qkv, ld_qkv, p, stream);
}

}  // namespace xclip
