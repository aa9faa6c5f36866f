// CTA-pair (cta_group::2) tcgen05 GEMM: one 256 x 256 output tile per 2-CTA cluster.
//
// CTA rank r stages rows [128 r, 128 r + 128) of the A tile and columns [128 r, 128 r + 128) of the
// B tile (32 KiB per k-block instead of 48 KiB for a 128 x 256 tile of its own); the leader CTA
// issues tcgen05.mma.cta_group::2 (M = 256, N = 256), which reads both CTAs' shared memory and
// writes each CTA's 128 accumulator rows into that CTA's TMEM.  With K = 512..768 the single-CTA
// kernel (gemm.cuh) is bound by L2 -> shared-memory operand traffic; the pair cuts it by a third
// (measured on a B200: 1176 -> 1373 TFLOP/s for [50176 x 768] x [2304 x 768]^T).
//
// Barriers: full[stage] lives in the LEADER (its arrive.expect_tx covers the 64 KiB both CTAs
// load; the peer's TMA credits the leader's barrier); empty[stage] and tmem_full[acc] are
// multicast-committed into both CTAs; tmem_empty[acc] lives in the leader and counts the
// epilogue warps of both CTAs.
//
// Epilogues (template parameter EPI):
//   PEPI_STORE   C = alpha*acc (+bias) (+residual): bf16 via TMA stores / fp32 / fp32 atomic
//   PEPI_FF_UP   feed-forward up-projection with GEGLU fused (x_clip/x_clip.py:180-183,191-192):
//                B is the up-projection weight with its rows permuted so that a tile holds the
//                value columns [128 t, 128 t + 128) and the MATCHING gate columns; writes
//                u = [value | gate] (reference layout, needed by the backward), hp = value *
//                gelu(gate) (bf16) and accumulates per-row (sum, sum^2) of bf16(hp).
//   PEPI_FF_DOWN feed-forward down-projection with the LayerNorm folded in (:193-195):
//                x2 = LN(hp) g W2^T + x1 = rstd_r (acc_rj - mean_r c_j) + x1_rj  with
//                acc = hp (W2 . g)^T and c_j = sum_k (W2 . g)_jk; also writes bf16(acc) and
//                (mean, rstd) for the backward.
//   PEPI_FF_BWD2 backward of LayerNorm(4d) + GEGLU fused into the down-projection's dgrad GEMM
//                gdh = dx (W2 . g): per element
//                  hn = (value*gelu(gate) - mean) rstd;  dhp = rstd (gdh - a_r - hn b_r)
//                  d value = dhp gelu(gate);  d gate = dhp value gelu'(gate)
//                with the two row means a_r = mean_k gdh, b_r = mean_k gdh*hn supplied by
//                xclip_ff_bwd_prep (they only need the d-wide vectors dx, W2g row sums and the saved
//                down-projection accumulator).  Reads u = [value | gate] by TMA one and a half steps
//                ahead, writes du - the [M, 4d] gradient dh never exists.
#pragma once

#include "gemm.cuh"

namespace xclip {

constexpr int PEPI_STORE = 0;
constexpr int PEPI_FF_UP = 1;
constexpr int PEPI_FF_DOWN = 2;
constexpr int PEPI_FF_BWD2 = 4;

template <int EPI>
struct PairCfg {
  // the GELU epilogues are latency-bound (two MUFU + a dependent polynomial per element): with two
  // warps per scheduler ncu showed 36 % issue-slot and 33 % XU utilisation while the tensor pipe idled
  // a third of the time, so they get four warps per scheduler
  static constexpr int kEpiWarps = (EPI == PEPI_FF_UP || EPI == PEPI_FF_BWD2) ? 16 : 4;
  static constexpr int kThreads = (kEpiWarps + 2) * 32;
  static constexpr int kABytes = kGemmBlockM * kGemmBlockK * 2;   // 16 KiB: this CTA's 128 rows of A
  static constexpr int kBBytes = 128 * kGemmBlockK * 2;           // 16 KiB: this CTA's 128 of 256 N columns
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBox = 128 * 128;                          // one [128 rows x 64 bf16] staging box
  // STORE: 2 boxes (double buffered); FF_UP: one box per column half (value, gate and hp pass through it
  // one after the other - they wait in registers; a second box per half was measured: it removes the
  // barrier stalls but costs the sixth mainloop stage, 0.366 -> 0.384 ms at K = 768); FF_DOWN: two
  // (out, acc) box pairs alternating by 64-column step; FF_BWD2: three SETS of (value, gate) boxes
  // rotate through "being loaded by TMA / worked on / being stored" - paid for with one mainloop stage
  // (with three stages the epilogue waited for the MMAs, with four it does not: the dgrad GEMM has
  // K = d <= 1024 and the kernel is bound by its epilogue)
  static constexpr int kStagingBytes =
      (EPI == PEPI_FF_BWD2 ? 6 : (EPI == PEPI_STORE || EPI == PEPI_FF_UP) ? 2 : 4) * kBox;
  static constexpr int kStages = EPI == PEPI_FF_BWD2 ? 4 : (EPI == PEPI_STORE || EPI == PEPI_FF_UP) ? 6 : 5;
  static constexpr int kBarrierBytes = 256;
  static constexpr int kScratchBytes = EPI == PEPI_FF_UP ? 2 * 128 * 8 : 0;   // row-sum exchange
  static constexpr int kTotal = kStages * kStageBytes + kStagingBytes + kBarrierBytes + kScratchBytes;
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, uint32_t smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void st_box_bf16x8(uint32_t box, int row, int chunk, const float* f) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(box + swz128(row, chunk)),
               "r"(pack_bf16x2(f[0], f[1])), "r"(pack_bf16x2(f[2], f[3])),
               "r"(pack_bf16x2(f[4], f[5])), "r"(pack_bf16x2(f[6], f[7]))
               : "memory");
}
__device__ __forceinline__ float bf16_rn(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

template <int A_MAJOR, int B_MAJOR, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(PairCfg<EPI>::kThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmC2,
                 const GemmParams p) {
  using S = PairCfg<EPI>;
  constexpr int kStages = S::kStages;
  constexpr int kEpiWarps = S::kEpiWarps;
  constexpr int BLOCK_N = 256;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * S::kABytes;
  uint8_t* smem_c = smem + kStages * S::kStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_c + S::kStagingBytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* tmem_full = bars + 2 * kStages;
  uint64_t* tmem_empty = bars + 2 * kStages + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;

  const int num_m2 = (p.M + 2 * kGemmBlockM - 1) / (2 * kGemmBlockM);
  const int num_n = (p.N + BLOCK_N - 1) / BLOCK_N;
  const int num_kb = (p.K + kGemmBlockK - 1) / kGemmBlockK;
  const int splits = p.split_k > 0 ? p.split_k : 1;
  const int kb_per_split = (num_kb + splits - 1) / splits;
  const int num_tiles = num_m2 * num_n * splits;

  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 2 * kEpiWarps);
    }
    if (EPI == PEPI_FF_BWD2)
      for (int i = 0; i < 3; ++i) mbar_init(&bars[16 + i], 1);     // u_full[set]
    fence_barrier_init();
  }
  if (warp == kEpiWarps && XCLIP_ONE_LANE(lane)) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI != PEPI_STORE || p.use_tma_store) tma_prefetch_desc(&tmC);
    if (EPI == PEPI_FF_UP || EPI == PEPI_FF_DOWN || EPI == PEPI_FF_BWD2) tma_prefetch_desc(&tmC2);
  }
  if (warp == kEpiWarps + 1) tmem_alloc_pair_512(tmem_slot);
  tcgen05_fence_before();
  cluster_sync_all();             // barriers of BOTH CTAs are initialised before any remote arrive
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kEpiWarps) {
    // ===================== TMA producer (both CTAs) =====================
    if (XCLIP_ONE_LANE(lane)) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = pair; t < num_tiles; t += npairs) {
        const int tmn = t % (num_n * num_m2);
        const int n_blk = tmn % num_n;
        const int m_blk = (tmn / num_n) * 2 + (int)rank;
        const int n0 = n_blk * BLOCK_N + (int)rank * 128;
        const int split = t / (num_n * num_m2);
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, num_kb);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * S::kStageBytes);
          uint8_t* sa = smem_a + stage * S::kABytes;
          uint8_t* sb = smem_b + stage * S::kBBytes;
          if (A_MAJOR == kMajorK) {
            tma_load_2d_pair(sa, &tmA, &full_bar[stage], kb * kGemmBlockK, m_blk * kGemmBlockM);
          } else {
#pragma unroll
            for (int g = 0; g < 2; ++g)
              tma_load_2d_pair(sa + g * (kGemmBlockK * 128), &tmA, &full_bar[stage],
                               m_blk * kGemmBlockM + g * 64, kb * kGemmBlockK);
          }
          if (B_MAJOR == kMajorK) {
            tma_load_2d_pair(sb, &tmB, &full_bar[stage], kb * kGemmBlockK, n0);
          } else {
#pragma unroll
            for (int g = 0; g < 2; ++g)
              tma_load_2d_pair(sb + g * (kGemmBlockK * 128), &tmB, &full_bar[stage], n0 + g * 64,
                               kb * kGemmBlockK);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kEpiWarps + 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {
      constexpr uint32_t idesc = make_idesc_bf16(2 * kGemmBlockM, BLOCK_N, A_MAJOR, B_MAJOR);
      constexpr uint32_t kLboMN = kGemmBlockK * 128;
      constexpr uint32_t kAStep = (A_MAJOR == kMajorK) ? 32u : 2048u;
      constexpr uint32_t kBStep = (B_MAJOR == kMajorK) ? 32u : 2048u;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int t = pair; t < num_tiles; t += npairs, ++it) {
        const int split = t / (num_n * num_m2);
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
            const uint64_t adesc = make_smem_desc(smem_u32(smem_a + stage * S::kABytes),
                                                  A_MAJOR == kMajorK ? 0u : kLboMN, 1024u);
            const uint64_t bdesc = make_smem_desc(smem_u32(smem_b + stage * S::kBBytes),
                                                  B_MAJOR == kMajorK ? 0u : kLboMN, 1024u);
#pragma unroll
            for (int k = 0; k < kGemmBlockK / 16; ++k)
              umma_bf16_pair(tmem_d, desc_advance(adesc, k * kAStep), desc_advance(bdesc, k * kBStep),
                             idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            umma_commit_pair(&empty_bar[stage]);
            if (kb == kb1 - 1) umma_commit_pair(&tmem_full[acc]);
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===================== epilogue (warps 0..kEpiWarps-1, both CTAs) =====================
    int it = 0;
    uint32_t store_count = 0;
    const int quarter = warp & 3;                 // TMEM lane quarter
    const int row_in_tile = quarter * 32 + lane;
    // ---- FF_BWD2 state: u_full barriers, the TMA load of one step's (value, gate) boxes, row scalars
    uint64_t* u_full = bars + 16;
    // step g of this CTA = 64-column group q = g & 3 of its (g >> 2)-th tile; box set g % 3
    auto load_u = [&](int g) {
      const int tmn_ = (pair + (g >> 2) * npairs) % (num_n * num_m2);
      const int kq_ = (tmn_ % num_n) * BLOCK_N + (g & 3) * 64;
      const int r0_ = ((tmn_ / num_n) * 2 + (int)rank) * kGemmBlockM;
      uint8_t* dst = smem_c + (g % 3) * 2 * S::kBox;
      uint64_t* bar = &u_full[g % 3];
      mbar_arrive_expect_tx(bar, 2 * S::kBox);
      tma_load_2d(dst, &tmC2, bar, kq_, r0_);                         // u[:, k ..]        value
      tma_load_2d(dst + S::kBox, &tmC2, bar, p.ff_hidden + kq_, r0_);  // u[:, 4d + k ..]   gate
    };
    const int my_steps = pair < num_tiles ? 4 * ((num_tiles - pair + npairs - 1) / npairs) : 0;
    float2 nst = make_float2(0.f, 0.f), nab = make_float2(0.f, 0.f);   // (mean, rstd), (a, b) of the NEXT tile's row
    auto load_row_scalars = [&](int tile) {
      nst = make_float2(0.f, 0.f); nab = make_float2(0.f, 0.f);
      if (tile < num_tiles) {
        const int tmn_ = tile % (num_n * num_m2);
        const int r_ = ((tmn_ / num_n) * 2 + (int)rank) * kGemmBlockM + row_in_tile;
        if (r_ < p.M) {
          nst = __ldg(reinterpret_cast<const float2*>(p.ff_stats + 2ll * r_));
          nab = __ldg(reinterpret_cast<const float2*>(p.ff_ab + 2ll * r_));
        }
      }
    };
    if constexpr (EPI == PEPI_FF_BWD2) {
      if (threadIdx.x == 0 && my_steps > 0) {       // steps 0 and 1 (a CTA with a tile has four steps)
        load_u(0);
        load_u(1);
      }
      load_row_scalars(pair);
    }
    for (int t = pair; t < num_tiles; t += npairs, ++it) {
      const int tmn = t % (num_n * num_m2);
      const int n_blk = tmn % num_n;
      const int m_blk = (tmn / num_n) * 2 + (int)rank;
      const int split = t / (num_n * num_m2);
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tmem_full[acc], acc_phase);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + acc * BLOCK_N;
      const int row = m_blk * kGemmBlockM + row_in_tile;
      const bool row_ok = row < p.M;
      if constexpr (EPI == PEPI_STORE) {
        gemm_epilogue_store<BLOCK_N>(p, tmC, smem_c, taddr, warp, lane, m_blk, n_blk, split, store_count);
      } else if constexpr (EPI == PEPI_FF_UP) {
        // accumulator columns [0,128) = value, [128,256) = gate of hidden units [128 n_blk, +128).
        // 16 warps: sub = warp>>2 owns hidden columns [32 sub, +32); subs {0,1} / {2,3} share one set
        // of (value, gate, hp) boxes [128 rows x 64 columns].
        const int sub = warp >> 2;
        const int bs = sub >> 1;                                      // box set
        const uint32_t stg = smem_u32(smem_c) + bs * S::kBox;         // this column half's staging box
        const bool issuer = (threadIdx.x == bs * 256);
        // All arithmetic happens BEFORE the staging boxes are touched: the results wait in registers
        // (48 packed words) while the previous tile's TMA stores are still draining the boxes, so the
        // store latency overlaps the TMEM reads and the GELU math instead of serialising with them.
        // (packed fp32x2 arithmetic: two columns per instruction, see common.cuh)
        float s1 = 0.f, s2 = 0.f;
        f32x2 s1p = f2_splat(0.f), s2p = f2_splat(0.f);
        uint32_t pv[16], pg[16], ph[16];
#pragma unroll
        for (int c16 = 0; c16 < 2; ++c16) {
          uint32_t vv[16], gg[16];
          tmem_ld_32x16(taddr + sub * 32 + c16 * 16, vv);
          tmem_ld_32x16(taddr + 128 + sub * 32 + c16 * 16, gg);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float va0 = __uint_as_float(vv[i]), va1 = __uint_as_float(vv[i + 1]);
            const float ga0 = __uint_as_float(gg[i]), ga1 = __uint_as_float(gg[i + 1]);
            const GeluParts2 gp = gelu_parts2(ga0, ga1);
            const f32x2 ge = f2_mul(f2_pack(ga0, ga1), gp.cdf);               // gelu(gate)
            const uint32_t hw = f2_to_bf16x2(f2_mul(f2_pack(va0, va1), ge));    // hp, rounded to bf16
            const f32x2 hr = f2_from_bf16x2(hw);           // statistics of what the next GEMM reads
            s1p = f2_add(s1p, hr);
            s2p = f2_fma(hr, hr, s2p);
            pv[c16 * 8 + (i >> 1)] = pack_bf16x2(va0, va1);
            pg[c16 * 8 + (i >> 1)] = pack_bf16x2(ga0, ga1);
            ph[c16 * 8 + (i >> 1)] = hw;
          }
        }
        {
          float a, b;
          f2_unpack(s1p, a, b); s1 = a + b;
          f2_unpack(s2p, a, b); s2 = a + b;
        }
        // the accumulator is in registers now: hand the TMEM buffer back to the MMA warp at once
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
        // the two warps sharing a row of this box set combine their partial sums (one red pair per
        // row, box set and tile instead of two)
        float2* xch = reinterpret_cast<float2*>(smem_c + S::kStagingBytes + S::kBarrierBytes) + bs * 128;
        if (sub & 1) xch[row_in_tile] = make_float2(s1, s2);
        // value, gate and hp pass through the single box one after the other
        const int hcol = n_blk * 128 + bs * 64;               // hidden-unit column of this box
        const int r0 = m_blk * kGemmBlockM;
#pragma unroll
        for (int which = p.ff_skip_u ? 2 : 0; which < 3; ++which) {
          if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          asm volatile("bar.sync %0, 256;" ::"r"(1 + bs) : "memory");
          const uint32_t* src = which == 0 ? pv : (which == 1 ? pg : ph);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t off = swz128(row_in_tile, (sub & 1) * 4 + c);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + off), "r"(src[4 * c]),
                         "r"(src[4 * c + 1]), "r"(src[4 * c + 2]), "r"(src[4 * c + 3]) : "memory");
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync %0, 256;" ::"r"(1 + bs) : "memory");
          if (issuer) {
            if (which == 0) tma_store_2d(&tmC, stg, hcol, r0);                      // u[:, hcol ..]       value
            else if (which == 1) tma_store_2d(&tmC, stg, p.ff_hidden + hcol, r0);   // u[:, 4d + hcol ..]  gate
            else tma_store_2d(&tmC2, stg, hcol, r0);                                // hp[:, hcol ..]
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
        if (!(sub & 1)) {
          const float2 o = xch[row_in_tile];
          s1 += o.x;
          s2 += o.y;
        }
        // one (sum, sum^2) slot per row and 64-column box: plain stores, summed in a fixed order by
        // the down-projection -> the statistics (and the loss) are bit-reproducible run to run
        if (row_ok && !(sub & 1)) {
          const int nparts = p.ff_hidden >> 6;                     // 4d / 64 boxes per row
          *reinterpret_cast<float2*>(p.ff_rowsum + 2ll * ((long long)row * nparts + n_blk * 2 + bs)) =
              make_float2(s1, s2);
        }
      } else if constexpr (EPI == PEPI_FF_BWD2) {
        // u is not fetched by ld.global -> st.shared at the start of each 64-column step: the warps then
        // sit on the HBM latency (ncu: 26 % long-scoreboard at the STS + 22 % barrier stalls behind it;
        // 0.346 vs 0.297 ms at [50176 x 768]).  Instead all 16 warps work on one 64-column step at a
        // time (a warp: its 32-row lane quarter x 16 columns) and a step's (value, gate) boxes arrive by
        // TMA in one of THREE box sets, requested one and a half steps ahead by thread 0 as soon as the
        // set's previous gradient store has been read:
        //   step g uses set g % 3;   L(g) = TMA load of step g;   S(g) = TMA store of step g
        //   prologue: L(0), L(1);    middle of step g: wait S(<= g-1) read, issue L(g+2)
        // The gradients overwrite u in place and leave by TMA store.
        const int cs = warp >> 2;                                      // which 16 columns of the 64-column step
        const bool issuer = threadIdx.x == 0;
        const float mean = nst.x, rstd = nst.y, am = nab.x, bm = nab.y;
        load_row_scalars(t + npairs);                                  // next tile's scalars travel during this one
        const f32x2 rstd2 = f2_splat(rstd), nmr = f2_splat(-mean * rstd), namr = f2_splat(-am * rstd),
                    nbmr = f2_splat(-bm * rstd);
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {
          const int g = 4 * it + q;
          const int set = g % 3;
          const int kq = n_blk * BLOCK_N + q * 64;
          const uint32_t stg = smem_u32(smem_c) + set * 2 * S::kBox;   // value -> d value | gate -> d gate
          mbar_wait(&u_full[set], (g / 3) & 1);
          uint32_t v[16];
          tmem_ld_32x16(taddr + q * 64 + cs * 16, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; i += 8) {
            if (i == 8 && issuer && g + 2 < my_steps) {
              // set (g+2) % 3 = (g-1) % 3: its store was committed half a step ago and has been read by now
              if (g >= 1) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
              load_u(g + 2);
            }
            const int chunk = cs * 2 + (i >> 3);
            const uint32_t off = swz128(row_in_tile, chunk);
            uint32_t wv[4], wg[4];
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(wv[0]), "=r"(wv[1]), "=r"(wv[2]), "=r"(wv[3]) : "r"(stg + off));
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(wg[0]), "=r"(wg[1]), "=r"(wg[2]), "=r"(wg[3]) : "r"(stg + S::kBox + off));
            uint32_t dvw[4], dgw[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {                           // two columns per step (fp32x2)
              const float g0 = __uint_as_float(wg[k] << 16), g1 = __uint_as_float(wg[k] & 0xffff0000u);
              const f32x2 gate = f2_pack(g0, g1), val = f2_from_bf16x2(wv[k]);
              const GeluParts2 gp = gelu_parts2(g0, g1);
              const f32x2 ge = f2_mul(gate, gp.cdf);                // gelu(gate)
              const f32x2 gd = f2_fma(gate, gp.pdf, gp.cdf);        // gelu'(gate)
              const f32x2 hn = f2_fma(f2_mul(val, ge), rstd2, nmr); // (val*ge - mean) rstd
              f32x2 dhp = f2_fma(f2_pack(__uint_as_float(v[i + 2 * k]), __uint_as_float(v[i + 2 * k + 1])),
                                 rstd2, namr);                      // rstd (gdh - a)
              dhp = f2_fma(hn, nbmr, dhp);                          //   - rstd b hn
              dvw[k] = f2_to_bf16x2(f2_mul(dhp, ge));
              dgw[k] = f2_to_bf16x2(f2_mul(f2_mul(dhp, val), gd));
            }
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + off), "r"(dvw[0]),
                         "r"(dvw[1]), "r"(dvw[2]), "r"(dvw[3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + S::kBox + off), "r"(dgw[0]),
                         "r"(dgw[1]), "r"(dgw[2]), "r"(dgw[3]) : "memory");
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 512;" ::: "memory");
          if (issuer) {
            const int r0 = m_blk * kGemmBlockM;
            tma_store_2d(&tmC, stg, kq, r0);                            // du[:, k ..]        d value
            tma_store_2d(&tmC, stg + S::kBox, p.ff_hidden + kq, r0);    // du[:, 4d + k ..]   d gate
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      } else {   // PEPI_FF_DOWN
        const uint32_t stg_base = smem_u32(smem_c);             // two (out box | acc box) pairs, alternating
        const float invD = 1.f / (float)p.ff_hidden;
        float mean = 0.f, rstd = 0.f;
        if (row_ok) {
          const int nparts = p.ff_hidden >> 6;
          const float4* parts = reinterpret_cast<const float4*>(p.ff_rowsum + 2ll * (long long)row * nparts);
          float sx = 0.f, sy = 0.f;
          for (int k = 0; k < nparts / 2; ++k) {                   // fixed order
            const float4 v = __ldg(parts + k);
            sx += v.x; sy += v.y; sx += v.z; sy += v.w;
          }
          mean = sx * invD;
          rstd = rsqrtf(fmaxf(sy * invD - mean * mean, 0.f) + p.ff_eps);
          if (n_blk == 0) *reinterpret_cast<float2*>(p.ff_stats + 2ll * row) = make_float2(mean, rstd);
        }
        const bf16* res_row = (p.residual != nullptr && row_ok) ? p.residual + (long long)row * p.ldr : nullptr;
#pragma unroll 1
        for (int q = 0; q < BLOCK_N / 64; ++q) {
          // this step's pair was last handed to TMA two steps ago: at most the previous step's group may
          // still be pending when it is rewritten
          const uint32_t stg = stg_base + (q & 1) * 2 * S::kBox;
          if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
          for (int c32 = 0; c32 < 2; ++c32) {
            uint32_t v[32];
            tmem_ld_32x32(taddr + q * 64 + c32 * 32, v);
            tmem_ld_wait();
            const int col0 = n_blk * BLOCK_N + q * 64 + c32 * 32;
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              float a8[8], o8[8];
              float r8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
              if (res_row != nullptr && col0 + i < p.N) {
                const uint4 r4 = *reinterpret_cast<const uint4*>(res_row + col0 + i);
                float2 x0 = unpack_bf16x2(r4.x), x1 = unpack_bf16x2(r4.y);
                float2 x2 = unpack_bf16x2(r4.z), x3 = unpack_bf16x2(r4.w);
                r8[0] = x0.x; r8[1] = x0.y; r8[2] = x1.x; r8[3] = x1.y;
                r8[4] = x2.x; r8[5] = x2.y; r8[6] = x3.x; r8[7] = x3.y;
              }
              float c8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
              if (col0 + i < p.N) {
                const float4 c0 = *reinterpret_cast<const float4*>(p.ff_colvec + col0 + i);
                const float4 c1 = *reinterpret_cast<const float4*>(p.ff_colvec + col0 + i + 4);
                c8[0] = c0.x; c8[1] = c0.y; c8[2] = c0.z; c8[3] = c0.w;
                c8[4] = c1.x; c8[5] = c1.y; c8[6] = c1.z; c8[7] = c1.w;
              }
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                a8[e] = __uint_as_float(v[i + e]);
                o8[e] = fmaf(rstd, a8[e] - mean * c8[e], r8[e]);
              }
              const int chunk = c32 * 4 + (i >> 3);
              st_box_bf16x8(stg, row_in_tile, chunk, o8);
              st_box_bf16x8(stg + S::kBox, row_in_tile, chunk, a8);
            }
          }
          fence_proxy_async_smem();
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (threadIdx.x == 0) {
            const int c0 = n_blk * BLOCK_N + q * 64;
            if (c0 < p.N) {
              tma_store_2d(&tmC, stg, c0, m_blk * kGemmBlockM);
              tma_store_2d(&tmC2, stg + S::kBox, c0, m_blk * kGemmBlockM);
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      if constexpr (EPI != PEPI_FF_UP) {     // (FF_UP released its accumulator before staging)
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
      }
    }
    // outstanding TMA stores must have READ their staging smem before the CTA exits
    if (EPI == PEPI_FF_UP || EPI == PEPI_FF_BWD2) {
      if ((threadIdx.x & 255) == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    } else if ((EPI != PEPI_STORE || p.use_tma_store) && threadIdx.x == 0) {
      asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();             // nobody exits (or frees TMEM) while the peer may still signal it
  if (warp == kEpiWarps + 1) {
    tcgen05_fence_after();
    tmem_dealloc_pair_512(tmem_base);
  }
}

}  // namespace xclip
