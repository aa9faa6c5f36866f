/*
 * xclip_b200.h - C-ABI of the B200-native CLIP training hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b): plain `extern "C"` entry points,
 * raw device pointers + explicit shapes, a cudaStream_t, int return codes.  The
 * CALLER (PyTorch, through x_clip_b200/_lib.py) owns every buffer; the library
 * never allocates persistent device memory, never synchronises the host, never
 * throws and never exits.  All pointers are device pointers unless stated.
 *
 * Each entry point names the reference call site it replaces
 * (lucidrains/x-clip v0.14.4, paths relative to /root/reference).
 *
 * Conventions
 *   - "bf16" buffers hold __nv_bfloat16, "f32" buffers hold float.
 *   - Row-major everywhere; `ld*` are leading dimensions in ELEMENTS.
 *   - return 0 on success; otherwise an XCLIP_ERR_* code and xclip_last_error()
 *     returns a thread-local message.
 *   - Work is enqueued on `stream` and is asynchronous w.r.t. the host.
 */
#ifndef XCLIP_B200_H_
#define XCLIP_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define XCLIP_OK 0
#define XCLIP_ERR_INVALID 1      /* bad argument / unsupported shape */
#define XCLIP_ERR_CUDA 2         /* CUDA runtime / driver error */
#define XCLIP_ERR_UNSUPPORTED 3  /* device is not sm_100 */

#define XCLIP_MAJOR_K 0  /* operand stored with the contraction index contiguous */
#define XCLIP_MAJOR_MN 1 /* operand stored transposed (its M / N index contiguous) */

typedef void* xclip_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------- */
int xclip_abi_version(void);
const char* xclip_last_error(void);
/* Binds to the current CUDA device, checks it is sm_100, resolves the driver
 * entry point used for TMA descriptors.  Idempotent. */
int xclip_init(void);
/* number of kernels this library has launched since the last reset (host counter) */
long long xclip_launch_count(void);
void xclip_launch_count_reset(void);
/* Tuning switches: returns the previous value, -1 for an unknown knob.  No knobs are left, so every
 * call returns -1 and changes nothing (kept for callers of ABI version 1, e.g. bench.py --tune). */
int xclip_tune_set(int knob, int value);

/* ---- dense contraction (tcgen05) --------------------------------------
 * C[M,N] (+)= alpha * A * B^T (+ bias[N]) (+ residual[res_row_idx[row] | row % res_row_mod | row, N])
 * Replaces nn.Linear fwd + its autograd dgrad/wgrad:
 *   x_clip/x_clip.py:191,195 (FeedForward), :209,:210 (Attention to_qkv/to_out),
 *   :358 (patch embedding, with bias), :368 (to_cls_tokens), :556,:570 (latent proj).
 * a_major = K : A is [M,K] (lda >= K).   a_major = MN : A is stored as [K,M] (lda >= M).
 * b_major = K : B is [N,K] (ldb >= K) - the nn.Linear [out,in] layout.
 * b_major = MN: B is stored as [K,N] (ldb >= N).
 * c_dtype 0 = bf16, 1 = f32.  accumulate != 0 (f32 only): C += result (atomic; enables
 * split-K over `K` when the output has too few tiles to fill the GPU - the wgrad case).
 * Requirements: N % 8 == 0, lda/ldb/ldr % 8 == 0, ldc % 8 == 0 (bf16) or % 4 (f32),
 * 16-byte aligned base pointers.  bias is f32, residual is bf16.
 */
/* 256-wide problems run on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles) by default;
 * xclip_gemm_set_pair_mode(0) selects the single-CTA 128 x 256 kernel instead (returns the
 * previous setting).  Same results either way - a tuning / A-B switch, process-wide. */
int xclip_gemm_set_pair_mode(int enabled);
int xclip_gemm_bf16(const void* a, int64_t lda, int a_major, const void* b, int64_t ldb,
                    int b_major, void* c, int64_t ldc, int c_dtype, int M, int N, int K,
                    float alpha, const float* bias, const void* residual, int64_t ldr,
                    int res_row_mod, const int32_t* res_row_idx, int accumulate,
                    xclip_stream_t stream);

/* ---- row-wise kernels ---------------------------------------------------
 * Gain-only LayerNorm, biased variance (x_clip/x_clip.py:112-121).  One call can also apply
 * the residual add of the block (:288) and the NEXT pre-norm (:126) so the row is read once:
 *   out  = LN(x) * g (+ res)                      stats  = (mean, rstd) of x        [rows,2] f32
 *   out2 = LN(bf16(out)) * g2   (if g2 != NULL)   stats2 = (mean, rstd) of bf16(out)
 * x/res/out/out2 bf16 [rows, d]; g/g2 f32 [d]; d in 256*{1,2,3,4}.  eps: the reference uses
 * 1e-5 for fp32 activations and 1e-3 otherwise (:118) - the caller chooses. */
int xclip_layernorm_fwd(const void* x, int64_t ldx, const float* g, const void* res,
                        int64_t ldres, void* out, int64_t ldo, float* stats, const float* g2,
                        void* out2, int64_t ldo2, float* stats2, int rows, int d, float eps,
                        xclip_stream_t stream);
/* dx = dLN(dy; x, stats, g) (+ add);  dg += sum_rows dy * xhat   (dg f32 [d], accumulated) */
int xclip_layernorm_bwd(const void* dy, int64_t lddy, const void* x, int64_t ldx,
                        const float* stats, const float* g, const void* add, int64_t ldadd,
                        void* dx, int64_t lddx, float* dg, int rows, int d,
                        xclip_stream_t stream);
/* l2norm = F.normalize(dim=-1, eps=1e-12) (x_clip/x_clip.py:54-55, used at :715,:724).
 * p f32 [rows,d] -> z f32 [rows,d], inv = 1/max(|p|,eps), and the split-bf16 operands of the
 * logits contraction: zrow = [hi|lo|hi], zcol = [hi|hi|lo], bf16 [rows,3d], hi = bf16(z),
 * lo = bf16(z - hi).  zrow . zcol^T = hi.hi + lo.hi + hi.lo matches the fp32 dot product to
 * ~2^-17, so the logits keep fp32-level accuracy while running on the bf16 tensor cores. */
int xclip_l2norm_fwd(const float* p, int64_t ldp, float* z, void* zrow, void* zcol, float* inv,
                     int rows, int d, xclip_stream_t stream);
/* dp (bf16) = inv * (dz - z <z,dz>) */
int xclip_l2norm_bwd(const float* dz, const float* z, const float* inv, void* dp, int rows, int d,
                     xclip_stream_t stream);
int xclip_cast_f32_bf16(const float* src, void* dst, int64_t n, xclip_stream_t stream);

/* ---- fused attention (tcgen05) -------------------------------------------
 * Attention core of x_clip/x_clip.py:217-244 (dim_head = 64, n <= 320).  causal != 0 adds the
 * reference's causal mask (keys j > i get -FLT_MAX, :233-236); implemented for n <= 128.
 * qkv bf16 [B*n, ld_qkv] holds q | k | v, each heads*64 wide, head-major inside.
 * key_mask uint8 [B, n] (1 = attend; may be NULL).  o bf16 [B*n, ldo] (heads merged).
 * lse f32 [B, heads, n]: base-2 log-sum-exp of scale*log2(e)*scores (saved for backward). */
int xclip_attn_fwd(const void* qkv, int64_t ld_qkv, const uint8_t* key_mask, void* o, int64_t ldo,
                   float* lse, int B, int n, int heads, float scale, int causal,
                   xclip_stream_t stream);
/* delta f32 [B, heads, n] is scratch (rowsum(dO*O), written here).  dq_workspace f32
 * [B*n, heads*64] is required when n > 128 (partial dQ across key tiles), else may be NULL;
 * its contents are scratch too (with XCLIP_ATTN_TAIL=1 and n = 128k+1 the first three floats of a
 * token's 64-float slot also carry the tail-token scalars between the two backward kernels). */
int xclip_attn_bwd(const void* qkv, int64_t ld_qkv, const uint8_t* key_mask, const void* o,
                   int64_t ldo, const void* d_o, int64_t lddo, const float* lse, float* delta,
                   void* dqkv, int64_t ld_dqkv, float* dq_workspace, int B, int n, int heads,
                   float scale, int causal, xclip_stream_t stream);

/* ---- similarity + InfoNCE / DCL (tcgen05, logits never materialised in forward) ----------
 * Replaces x_clip/x_clip.py:813-847 for one direction of the loss:
 *   s[r,c] = *temp_exp * <a_r, b_c> (temp_exp: DEVICE scalar exp(temperature), so the host
 *   never synchronises on the parameter),  a bf16 [R,D] = LOCAL unit-norm latents of one modality,
 *   b bf16 [C,D] = ALL latents of the other modality; the positive of row r is column
 *   r + diag_offset.  dcl != 0 removes the positive from the denominator (:834-836).
 * fwd:  lse[r] = log sum_c exp(s[r,c]);  pos[r] = s[r, r+diag_offset];
 *       *loss_accum += loss_scale * sum_r (lse[r] - pos[r])     (loss_accum may be NULL)
 *       part_ws: f32 scratch [2 * xclip_nce_num_col_blocks(C) * R] (per block: max, sum; the
 *       log-sum-exp uses an online maximum, so any temperature works).
 *       (the reference's +1e-20 inside its logs, :51-52, is below fp32 resolution here)
 * bwd:  g[r,c] = *gscale * (w_row*exp(s - lse_row[r]) + w_col*exp(s - lse_col[c])
 *                           - w_diag*[c == r+diag])     (gscale: DEVICE scalar, upstream grad
 *       / (2*B_global); exp terms skipped on the positive when dcl).  Written as
 *       bf16 temp_exp*g [R, ldg>=roundup8(C)], so the latent gradient is dA = (that) @ b via
 *       xclip_gemm_bf16;  *dtemp += sum g*s (d loss / d temperature) when dtemp != NULL. */
int xclip_nce_num_col_blocks(int C);
int xclip_nce_fwd(const void* a, const void* b, int R, int C, int D, const float* temp_exp,
                  int diag_offset, int dcl, float* part_ws, float* pos, float* lse,
                  float* loss_accum, float loss_scale, xclip_stream_t stream);
int xclip_nce_bwd(const void* a, const void* b, int R, int C, int D, const float* temp_exp,
                  int diag_offset, int dcl, const float* lse_row, const float* lse_col,
                  float w_row, float w_col, float w_diag, const float* gscale, void* g,
                  int64_t ldg, float* dtemp, xclip_stream_t stream);

/* ---- FILIP fine-grained loss (x_clip/x_clip.py:799-811 + :821-847) -----------------------
 * segmax : a bf16 [R,D] token latents of one modality, b bf16 [C,D] token latents of the other,
 *          C = n_samples * seg_len (seg_len tokens per sample, multiple of 16, <= 256).  For
 *          every row r and sample y: seg_max[r,y] = max_i s, seg_arg[r,y] = argmax_i s with
 *          s = *temp_exp * <a_r, b_(y,i)> (optionally s*col_mul[c] + col_add[c]: padded text
 *          tokens get col_mul 0 / col_add -FLT_MAX, the reference's masked_fill at :810).
 * reduce : out[a,b] = sum_k weights[a*len+k] * seg_max[(a*len+k), b]  ([samples, nseg] or
 *          transposed) - the masked mean over text tokens (:807) / mean over image tokens (:811).
 * nce_fwd/bwd : row-wise InfoNCE / DCL on an [R,C] fp32 similarity matrix (R local texts, C all
 *          images, positive of row x at column x + diag_off) (:821-847); bwd writes
 *          g = *gscale * (softmax_row - [positive]).
 * expand : rows [row0,row0+rows) of the backward operand G[R,C] (bf16): at the argmax column
 *          of each (row, sample) the value *temp_exp * wmat[row/rows_per_sample, sample] *
 *          rowscale[row], zero elsewhere; *dtemp += sum w * seg_max.  d rows = G @ b and
 *          d cols += G^T @ a then run on xclip_gemm_bf16. */
int xclip_filip_segmax(const void* a, const void* b, int R, int C, int D, const float* temp_exp,
                       int seg_len, const float* col_mul, const float* col_add, float* seg_max,
                       int* seg_arg, xclip_stream_t stream);
int xclip_filip_reduce(const float* seg_max, const float* weights, int samples, int len, int nseg,
                       float* out, int transpose_out, xclip_stream_t stream);
int xclip_filip_nce_fwd(const float* s, int R, int C, int diag_off, int dcl, float* lse,
                        float* loss_accum, float loss_scale, xclip_stream_t stream);
int xclip_filip_nce_bwd(const float* s, const float* lse, int R, int C, int diag_off, int dcl,
                        const float* gscale, float* g, xclip_stream_t stream);
int xclip_filip_expand(const int* seg_arg, const float* seg_max, const float* wmat,
                       const float* rowscale, const float* temp_exp, int row0, int rows,
                       int rows_per_sample, int seg_len, int nseg, void* g, int64_t ldg,
                       float* dtemp, xclip_stream_t stream);

/* ---- text embedding (x_clip/x_clip.py:320-332) ---------------------------------------------
 * fwd: out bf16 [B, n+1, d]: out[b,0] = cls, out[b,1+t] = tok[ids[b,t]] + pos[t]  (fp32 tables,
 *      ids int64 [B,n]; an id outside [0, vocab) traps the kernel - the launch
 *      fails like nn.Embedding's device-side assert, nothing is clamped silently).
 * bwd: dx bf16 [B, n+1, d] -> dtok f32 [vocab,d] (+=, vector reductions), dpos f32 [>=n, d] (+=),
 *      dcls f32 [d] (+=).  All three gradients must be zero-initialised by the caller. */
int xclip_text_embed_fwd(const int64_t* ids, const float* tok, const float* pos, const float* cls,
                         void* out, int B, int n, int d, int vocab, xclip_stream_t stream);
int xclip_text_embed_bwd(const int64_t* ids, const void* dx, float* dtok, float* dpos, float* dcls,
                         int B, int n, int d, int vocab, xclip_stream_t stream);

/* ---- fused feed-forward block (x_clip/x_clip.py:180-199) on the CTA-pair GEMM ------------------
 * FeedForward = Linear(d, 8d) -> GEGLU -> LayerNorm(4d) -> Linear(4d, d), + residual (:289).
 *   ff_permute_cast : bf16 copy of net.0.weight [8d, d] with rows reordered so that a 256-row tile
 *                     holds 128 value rows and the 128 MATCHING gate rows.
 *   ff_scale_cast   : w2g = bf16(net.4.weight [d, 4d] * net.2.g [4d]) and colvec[j] = sum_k w2g[j,k].
 *   ff_up           : u = [value | gate] bf16 [M, 8d] (reference layout, kept for the backward),
 *                     hp = value * gelu_erf(gate) bf16 [M, 4d], rowsum[r, box] = (sum hp, sum hp^2) of
 *                     every 64-column box (rowsum f32 [M, 4d/64, 2], fully overwritten: no atomics,
 *                     bit-reproducible) - one GEMM, GEGLU in its epilogue.
 *                     u may be NULL (forward-only sweeps: two thirds of the output traffic saved).
 *   ff_down         : (mean_r, rstd_r) from rowsum; out = rstd_r * (hp w2g^T - mean_r * colvec) + residual
 *                     (== LN(hp) g W2^T + x1),
 *                     acc_out = bf16(hp w2g^T), stats[r] = (mean, rstd) - one GEMM.
 *   ff_bwd_prep     : dxs = bf16(dx * rstd_r) [M, d]; vsum[j] += sum_r dxs[r,j] * mean_r; with acc and
 *                     colvec also ab[r] = (mean_k gdh, mean_k gdh*hn) - the two row means of the
 *                     LayerNorm backward, from d-wide data only (gdh = dx w2g is never formed here).
 *   ff_bwd          : du [M, 8d] = backward of LayerNorm(4d) + GEGLU fused into the dgrad GEMM
 *                     gdh = dx w2g (reads u, stats, ab; the [M, 4d] gradient never exists in HBM).
 *   ff_w2_grad_post : in place on raw = dxs^T hp (f32 [d, 4d]): dW2[j,k] = g[k] * (raw[j,k] - vsum[j]);
 *                     with w2/dg also dg[k] += sum_j (raw[j,k] - vsum[j]) * w2[j,k] (gain gradient).
 * d in 256*{1,2,3,4}; all matrices row-major, bf16 unless stated. */
int xclip_ff_permute_cast(const float* w1, void* out, int d, xclip_stream_t stream);
int xclip_ff_scale_cast(const float* w2, const float* g, void* w2g, float* colvec, int d,
                        xclip_stream_t stream);
int xclip_ff_up(const void* x, int64_t ldx, const void* w1p, void* u, int64_t ldu, void* hp,
                int64_t ldhp, float* rowsum, int M, int d, xclip_stream_t stream);
int xclip_ff_down(const void* hp, int64_t ldhp, const void* w2g, const float* colvec,
                  const float* rowsum, const void* residual, int64_t ldr, void* out, int64_t ldo,
                  void* acc_out, int64_t ldacc, float* stats, float eps, int M, int d,
                  xclip_stream_t stream);
int xclip_ff_bwd_prep(const void* dx, int64_t lddx, const float* stats, const void* acc, int64_t ldacc,
                      const float* colvec, void* dxs, float* vsum, float* ab, int rows, int d,
                      xclip_stream_t stream);
int xclip_ff_bwd(const void* dx, int64_t lddx, const void* w2g, const void* u, int64_t ldu,
                 const float* stats, const float* ab, void* du, int64_t lddu, int M, int d,
                 xclip_stream_t stream);
int xclip_ff_w2_grad_post(float* raw, const float* vsum, const float* g, const float* w2, float* dg,
                          int d, xclip_stream_t stream);

/* ---- fused AdamW (SURVEY 8f: the optimizer step behind the gradient all-reduce; the reference
 * leaves optimisation to the user, README.md:44-58) over one flat f32 buffer; identical update rule to
 * torch.optim.AdamW (decoupled decay, bias correction with `step` >= 1); g is read as g*grad_scale. */
int xclip_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                     float beta2, float eps, float weight_decay, int step, float grad_scale,
                     xclip_stream_t stream);

/* ---- patch-embedding front end (x_clip/x_clip.py:356-359 patchify, :134-151 PatchDropout) -------
 * patchify_gather : img f32 [B,C,H,W] -> bf16 [B*k, patch*patch*C] rows in the reference's
 *                   (p1 p2 c) order for the patches keep[b, j] (int64 [B,k]; NULL = all k = n patches,
 *                   in order): only kept patches are read and embedded.
 * scatter_add_rows: dst f32 [V,d] rows idx[r] (or r %% period) += src bf16 [rows,d]  (gradient of the
 *                   gathered position table);  colsum_rows: dst[d] += column sums (bias gradient). */
int xclip_patchify_gather(const float* img, int B, int C, int H, int W, int patch, const int64_t* keep,
                          int k, void* out, xclip_stream_t stream);
int xclip_scatter_add_rows(const int32_t* idx, int period, const void* src, int64_t lds, float* dst,
                           int64_t rows, int d, int V, xclip_stream_t stream);
int xclip_colsum_rows(const void* src, int64_t lds, float* dst, int64_t rows, int d,
                      xclip_stream_t stream);

/* ---- rotary position embedding (x_clip/x_clip.py:155-176, applied to q, k and v at :221-223) ----
 * In place on the bf16 qkv buffer [rows, ld] (rows = B*n tokens, position = row %% n): in each of
 * the `nslices` consecutive 64-wide head slices the first 32 features are rotated pairwise
 * (j with j+16) by angle[pos, j]; cos_tab / sin_tab f32 [n, 16].  inverse != 0: the transposed
 * rotation (backward, applied to dq | dk | dv). */
int xclip_rotary_inplace(void* qkv, int64_t ld, int64_t rows, int n, int nslices,
                         const float* cos_tab, const float* sin_tab, int inverse,
                         xclip_stream_t stream);

#ifdef __cplusplus
}
#endif

#endif /* XCLIP_B200_H_ */
