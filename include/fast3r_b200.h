/* fast3r_b200 — C ABI of the B200-native Fast3R forward-pass kernels (libfast3r_b200.so).
 *
 * Drop-in boundary for the single-forward-pass hot path of facebookresearch/fast3r
 * (CroCo encoder -> fusion decoder -> DPT heads).  The reference's only native precedent is the
 * `curope` torch extension (fast3r/croco/models/curope/curope.cpp:54-59, kernels.cu:84-108): free functions
 * over caller-owned device buffers, default/current stream, no ownership transfer, errors reported to Python
 * as RuntimeError.  This ABI keeps those conventions but is torch-free: plain pointers, sizes and a
 * cudaStream_t (passed as void*).  Every entry point
 *   - works on caller-owned DEVICE pointers (16-byte aligned), never allocates or synchronises,
 *   - enqueues on the given stream and returns 0 on success, non-zero on error (text via f3r_last_error()),
 *   - is reentrant per thread (one Python thread per GPU/process, like the reference).
 *
 * Layout conventions: activations are row-major "channels-last": a token / pixel is a row; bf16 unless noted.
 * Weights are bf16 [N_out, taps, K_in] (K contiguous); nn.Linear.weight (out,in) is already that with taps=1;
 * nn.Conv2d.weight (out,in,kh,kw) must be permuted to (out, kh*kw, in); ConvTranspose2d (in,out,k,k) to
 * ((i*k+j)*out + o, in).
 */
#ifndef FAST3R_B200_H
#define FAST3R_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define F3R_ABI_VERSION 2

/* epilogue kinds of f3r_gemm */
enum { F3R_EPI_STORE = 0, F3R_EPI_ROPE = 1, F3R_EPI_IDXEMB = 2, F3R_EPI_CONVT = 3, F3R_EPI_FINAL = 4 };
enum { F3R_ACT_NONE = 0, F3R_ACT_RELU = 1, F3R_ACT_GELU = 2 };

/* One fused GEMM / implicit-GEMM convolution:
 *   acc[m, n] = sum_{tap, k} A[pixel(m) + shift(tap), k] * Wt[n, tap, k]          (fp32 accumulation in TMEM)
 *   v = acc + bias[n] (+ RoPE2D | + idx-embedding row) (+ res0[m,n]) (+ res1[m,n])
 *   out1[m,n] = bf16(relu(v))   (optional);   out0[m,n] = act(v) as bf16 or fp32 (optional)
 * Replaces: nn.Linear qkv/proj/fc1/fc2 (fast3r/croco/models/blocks.py:94-97,125-128), decoder_embed + image-index
 * embedding add (fast3r/models/fast3r.py:782-799), RoPE2D on q,k (fast3r/croco/models/pos_embed.py:162-183),
 * patch-embed conv (blocks.py:412-414), every Conv2d/ConvTranspose2d of the DPT head
 * (fast3r/croco/models/dpt_block.py:42-77,105-123,187-195,367-381,416-481) and, with F3R_EPI_FINAL, the last
 * ReLU + conv1x1 + postprocess (dpt_block.py:378-381, fast3r/dust3r/heads/postprocess.py:16-64). */
typedef struct f3r_gemm_desc {
  const void* a;       /* bf16 activation, viewed as (nb, h, w, c) with pixel stride a_ld elements            */
  const void* wt;      /* bf16 weights [n, taps, k]                                                            */
  int32_t n, k, taps;  /* taps: 1 (linear / 1x1) or 9 (3x3, stride 1, zero pad 1)                              */
  int32_t w, h, nb;    /* spatial extent of A; a linear layer over M rows is (w=M, h=1, nb=1)                  */
  int32_t a_ld;        /* elements between consecutive pixels of A (>= k)                                      */
  int32_t epi, act;
  int32_t out0_f32, res0_f32;
  int32_t ldo;         /* row stride (elements) of out0 / out1 / res0 / res1                                   */
  int32_t split_col, ldo_b; /* columns >= split_col of out0 go to out0b (row stride ldo_b); 0 disables         */
  int32_t tok_per_img, grid_w, rope_cols; /* ROPE: tokens per image, patch-grid width, #leading columns rotated;
                                             IDXEMB: tok_per_img tokens share emb_ids[m / tok_per_img];
                                             tok_per_img == 0: one id per row, emb_ids[m]                     */
  int32_t ct_k, ct_cout;                  /* CONVT: kernel==stride k, out channels; n == k*k*ct_cout           */
  const float* bias;   /* [n] (CONVT: [ct_cout]) or NULL                                                       */
  const void* res0;    /* fp32 or bf16 [M, ldo] or NULL (may alias out0: in-place residual stream update)      */
  const void* res1;    /* bf16 [M, ldo] or NULL                                                                */
  void* out0;
  void* out0b;
  void* out1;
  const float* rope_cos; /* [max_pos, 16] cos(pos * base^(-j/16))                                              */
  const float* rope_sin;
  const float* emb_table; /* fp32 [1000, n]                                                                    */
  const int32_t* emb_ids; /* int32 [M / tok_per_img] (or [M] when tok_per_img == 0)                            */
  const float* w4;     /* FINAL: fp32 [4, n] 1x1 conv weight, b4 fp32 [4]                                      */
  const float* b4;
  float* pts;          /* FINAL: fp32 [M, 3]                                                                   */
  float* conf;         /* FINAL: fp32 [M]                                                                      */
} f3r_gemm_desc;

const char* f3r_last_error(void);
int f3r_abi_version(void);
/* sizeof(f3r_gemm_desc) as compiled into the library (binding-side struct layout guard). */
size_t f3r_gemm_desc_size(void);
/* Number of kernels launched through this library by the calling process so far. */
uint64_t f3r_launch_count(void);

/* Tuning knobs for A/B measurements (process-wide).  "attn_emu" = how many of every 8 exponential pairs of the
 * attention softmax are evaluated on the FMA pipe instead of MUFU.EX2 (0..3, -1 = built-in default); "attn_split" =
 * softmax threads per query row (1 or 2, -1 = default); "pdl" = 1 / 0: launch the GEMM / attention / LayerNorm chain with
 * programmatic dependent launch (successor prologues overlap predecessor tails; default 1, env F3R_PDL=0 disables). */
int f3r_set_option(const char* name, int32_t value);

int f3r_gemm(const f3r_gemm_desc* d, void* stream);

/* softmax(scale * Q K^T) V per (batch, head), head_dim 64, non-causal (blocks.py:135-194).
 * q: bf16 [batch, sq, ldq] (head h at columns h*64); kv: bf16 [batch, skv, ldkv] with K of head h at columns
 * h*64 and V at columns heads*64 + h*64; out: bf16 [batch, sq, ldo].  lse (optional): fp32 [batch, heads, sq]. */
int f3r_attention(const void* q, int32_t ldq, const void* kv, int32_t ldkv, void* out, int32_t ldo, float* lse,
                  int32_t batch, int32_t heads, int32_t sq, int32_t skv, float scale, void* stream);

/* Key-slice form of f3r_attention, for (a) filling the 148 SMs when batch*heads*ceil(sq/256) is small and (b) attending
 * to key ranges as they arrive over NVLink (sequence-parallel decoder, fast3r_b200/parallel.py): attends the queries to
 * the keys [kv_row0, kv_row0 + skv) of a kv buffer of kv_rows_total rows per batch, cut into n_split slices (one CTA each
 * per 256-row query tile); slice s writes its softmax-normalised fp32 output into part_o[part_base + s] (layout
 * [slot, batch*sq, heads*64]) and its log-sum-exp into part_lse[part_base + s] ([slot, batch, heads, sq]).
 * f3r_attention_merge combines n_parts slots into the exact softmax over the union of their keys (bf16 out). */
int f3r_attention_partial(const void* q, int32_t ldq, const void* kv, int32_t ldkv, int32_t kv_rows_total,
                          int32_t kv_row0, int32_t skv, int32_t n_split, float* part_o, float* part_lse,
                          int32_t part_base, int32_t batch, int32_t heads, int32_t sq, float scale, void* stream);
int f3r_attention_merge(const float* part_o, const float* part_lse, int32_t n_parts, void* out, int32_t ldo,
                        int32_t batch, int32_t heads, int32_t sq, void* stream);

/* nn.LayerNorm over the last dim of fp32 x [rows, dim] -> bf16 (or fp32) out  (blocks.py:219,228; fast3r.py:558,805) */
int f3r_layernorm(const float* x, const float* w, const float* b, void* out, int32_t out_f32, int32_t rows,
                  int32_t dim, float eps, void* stream);
/* fp32 image batch (n,3,H,W) -> bf16 (or, out_f32 != 0, fp32) [n*(H/16)*(W/16), 768] patch rows
 * (im2col of blocks.py:412 Conv2d k=s=16) */
int f3r_im2col_patch(const float* img, void* out, int32_t out_f32, int32_t n, int32_t h, int32_t w, void* stream);
/* bf16 NHWC (n,h,w,c) -> bf16 [n*ho*wo, 9*c] for the 3x3 stride-2 pad-1 conv (dpt_block.py:471-478) */
int f3r_im2col3x3s2(const void* in, void* out, int32_t n, int32_t h, int32_t w, int32_t c, int32_t ho, int32_t wo,
                    void* stream);
/* bilinear x2 align_corners=True on bf16 (f32 != 0: fp32) NHWC; writes the top-left (ho, wo) window of the (2h, 2w)
 * result (dpt_block.py:234-247,374; crop of dpt_head.py:69-71) */
int f3r_upsample2x(const void* in, void* out, int32_t f32, int32_t n, int32_t h, int32_t w, int32_t c, int32_t ho,
                   int32_t wo, void* stream);
/* fp32 -> bf16, count multiple of 4 */
int f3r_cast_bf16(const float* in, void* out, size_t count, void* stream);


/* ---- block-level entry: n_blocks consecutive transformer blocks (fast3r/croco/models/blocks.py:197-239) on the fp32
 * residual stream x [batch*seq, dim], in place:  x += proj(SDPA(rope(q), rope(k), v));  x += fc2(GELU(fc1(LN(x)))).
 * Composition of f3r_layernorm / f3r_gemm / f3r_attention (7 launches per block) with the operand buffers carved out of a
 * caller-owned workspace (f3r_transformer_workspace bytes, 256-byte aligned) - a C / C++ caller runs the CroCo encoder
 * (rope_cos != NULL: RoPE2D on q, k with positions from the patch grid) or a span of fusion-decoder blocks (rope_cos ==
 * NULL) with one call.  bf16 fast path, single device; attention over all seq keys of each batch element. */
typedef struct f3r_block_weights {
  const float* norm1_w; const float* norm1_b; const float* norm2_w; const float* norm2_b;   /* fp32 [dim]           */
  const void* qkv_w;  const float* qkv_b;   /* bf16 [3 dim, dim] rows ordered q | k | v (blocks.py:138-143), fp32 [3 dim] */
  const void* proj_w; const float* proj_b;  /* bf16 [dim, dim], fp32 [dim]                                           */
  const void* fc1_w;  const float* fc1_b;   /* bf16 [hidden, dim], fp32 [hidden]                                     */
  const void* fc2_w;  const float* fc2_b;   /* bf16 [dim, hidden], fp32 [dim]                                        */
} f3r_block_weights;
size_t f3r_transformer_workspace(int32_t rows, int32_t dim, int32_t hidden);
int f3r_transformer_blocks(const f3r_block_weights* blocks, int32_t n_blocks, float* x, int32_t batch, int32_t seq,
                           int32_t dim, int32_t heads, int32_t hidden, float eps, float scale, int32_t rope_grid_w,
                           int32_t rope_tok_per_img, const float* rope_cos, const float* rope_sin, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ---- image ingest (SURVEY §8 f3): PIL.Image.resize(LANCZOS | BICUBIC) + center crop + ToTensor + Normalize(0.5, 0.5) of
 * load_images() (fast3r/dust3r/utils/image.py:68-159) on a decoded 8-bit RGB image, bit-exact with Pillow's 8-bit
 * resampler.  filter: 0 = BICUBIC, 1 = LANCZOS.  f3r_resample_coeffs (HOST function, no CUDA call) fills the tap tables of
 * one dimension: bounds [out_size][2] = (first tap, count), kk [out_size][f3r_resample_ksize()] fixed-point weights, and
 * returns the widest source span of 64 consecutive outputs (h_span_max below; < 0 on error).  f3r_ingest_rgb8 takes DEVICE
 * copies of the tables (NULL for a dimension that keeps its size), a device scratch tmp [h][ow][3] (when ow != w) and
 * writes the crop box (left, top, cw, ch) of the resized image as fp32 [3][ch][cw] in [-1, 1]. */
int f3r_resample_ksize(int32_t in_size, int32_t out_size, int32_t filter);
int f3r_resample_coeffs(int32_t in_size, int32_t out_size, int32_t filter, int32_t* bounds, int32_t* kk);
int f3r_ingest_rgb8(const uint8_t* src, int32_t h, int32_t w, int32_t oh, int32_t ow, const int32_t* hb, const int32_t* hk,
                    int32_t hks, int32_t h_span_max, const int32_t* vb, const int32_t* vk, int32_t vks, uint8_t* tmp,
                    int32_t left, int32_t top, int32_t cw, int32_t ch, float* out, void* stream);

/* ---- geometry tail (SURVEY §8 f2, first slice): what every caller runs on the forward's outputs before poses.
 * A "view" below is one (view, batch item) pointmap of n = H*W pixels; all arrays are DEVICE pointers, fp32, view-major.
 *
 * f3r_conf_quantile: thr[v] = torch.quantile(conf[v].reshape(-1), q) (linear interpolation, fp32 like ATen) - the
 *   confidence threshold of align_local_pts3d_to_global (fast3r/models/multiview_dust3r_module.py:477) and of
 *   estimate_focal (:1093).  Exact: radix select on the float bit patterns.
 * f3r_similarity_fit: per view the least-squares similarity (R, t, s), y ~ s R x + t, over the pixels with
 *   conf >= thr & valid; fewer than 3 such pixels -> over valid only; still fewer -> identity (:480-515, where the fit is
 *   roma.rigid_points_registration(x, y, compute_scaling=True)).  conf/thr and valid may be NULL (no such mask).
 *   rts [views][13] = R row-major (9), t (3), s.  workspace: f3r_similarity_fit_workspace(views) bytes, 8-byte aligned.
 * f3r_similarity_apply: out = s (x R^T) + t on all n pixels of every view (:517-521).  out may alias x.
 * f3r_focal_weiszfeld: focal[v] = argmin_f sum |pixel - pp - f (x, y)/z| by `iters` IRLS steps from the L2 closed form,
 *   over the pixels with conf >= thr (conf/thr NULL: all pixels), clipped to [0, inf); no selected pixel -> max(H, W) /
 *   (2 tan 30 deg).  iters = 100 with a mask reproduces estimate_focal_knowing_depth_and_confidence_mask(weiszfeld)
 *   (fast3r/dust3r/post_process.py:82-142), iters = 10 without one estimate_focal_knowing_depth(weiszfeld) (:19-79).
 *   pts [views][H][W][3]; pp [views][2] or NULL (= (W/2, H/2)).  workspace: f3r_focal_workspace(views) bytes. */
int f3r_conf_quantile(const float* conf, int32_t views, int32_t n, float q, float* thr, void* stream);
size_t f3r_similarity_fit_workspace(int32_t views);
int f3r_similarity_fit(const float* x, const float* y, const float* conf, const float* thr, const uint8_t* valid,
                       int32_t views, int32_t n, float* rts, void* workspace, size_t workspace_bytes, void* stream);
int f3r_similarity_apply(const float* x, const float* rts, float* out, int32_t views, int32_t n, void* stream);
size_t f3r_focal_workspace(int32_t views);
int f3r_focal_weiszfeld(const float* pts, const float* conf, const float* thr, const float* pp, int32_t views, int32_t h,
                        int32_t w, int32_t iters, float* focal, void* workspace, size_t workspace_bytes, void* stream);

/* ---- camera poses (SURVEY §8 f2): fast_pnp (fast3r/dust3r/cloud_opt/init_im_poses.py:300-350), i.e. per view and per
 * candidate focal a RANSAC PnP over the masked pixels, for all views of one shape in one call.
 * pts [views][h][w][3] fp32 pointmap, mask [views][h][w] uint8 (non-zero: pixel used), focals [views][n_focals] fp32
 * candidates, pp [views][2] fp32 principal points or NULL (= (w/2, h/2)).  Pixel (x, y) is the point (x, y): integer
 * coordinates.  Per view and focal k, `iters` hypotheses i: 4 distinct masked pixels drawn by a fixed counter-based hash
 * of (k, i, draw), P3P on three, the fourth picks among its solutions.  scores [views][n_focals][iters] int32 = number of
 * masked pixels with reprojection error <= 5 px under the hypothesis, tested division-free in fp32 as
 * (P0 X - u P2 X)^2 + (P1 X - v P2 X)^2 <= 25 (P2 X)^2 with P = K [R | t] (a point with P2 X = 0 never counts).
 * best [views][2] = (k, i) of the highest score, ties to the lowest k then i, or (-1, -1) when every score is 0
 * (also when fewer than 4 pixels are masked).  The selected pose is refined by Levenberg-Marquardt steps on the
 * reprojection error over its inliers; c2w [views][3][4] fp64 = its camera-to-world inverse [R^T | -R^T t] (zeros for a
 * failed view).  workspace: f3r_pnp_workspace(views, h, w, n_focals, iters) bytes, 256-byte aligned.  Deterministic:
 * results depend neither on scheduling nor on which other views share the call. */
size_t f3r_pnp_workspace(int32_t views, int32_t h, int32_t w, int32_t n_focals, int32_t iters);
int f3r_pnp_ransac(const float* pts, const uint8_t* mask, int32_t views, int32_t h, int32_t w, const float* focals,
                   int32_t n_focals, const float* pp, int32_t iters, int32_t* scores, int32_t* best, double* c2w,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---- parity mode: the reference's fp32 path (inference_multiview.py:41-49, dtype="32": no autocast) on the bf16
 * tensor pipe.  Every fp32 operand x is carried as hi + lo (two bf16), every product as hi*hi + lo*hi + hi*lo with
 * fp32 accumulation.  For f3r_gemm this is the ordinary kernel over a 3x longer K: A' = f3r_split3(A) = [hi|lo|hi],
 * weights packed by the caller as [Whi | Whi | Wlo] along K (per tap); all outputs fp32 (out0_f32). */

/* fp32 in [rows, k] -> bf16 out [rows, 3k] = [hi | lo | hi] of x (relu != 0: of max(x, 0)) */
int f3r_split3(const float* in, void* out, size_t rows, int32_t k, int32_t relu, void* stream);
/* dst[i] += src[i], fp32, count multiple of 4 (second residual operand of dpt_block.py:241 in parity mode) */
int f3r_add_f32(float* dst, const float* src, size_t count, void* stream);
/* Same contract as f3r_attention with fp32 q / kv / out (blocks.py:135-194 without autocast).  workspace: caller-owned
 * device scratch of at least f3r_attention_x3_workspace() bytes, 256-byte aligned (holds the split operands). */
size_t f3r_attention_x3_workspace(int32_t batch, int32_t heads, int32_t sq, int32_t skv);
int f3r_attention_x3(const float* q, int32_t ldq, const float* kv, int32_t ldkv, float* out, int32_t ldo, float* lse,
                     void* workspace, size_t workspace_bytes, int32_t batch, int32_t heads, int32_t sq, int32_t skv,
                     float scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif
