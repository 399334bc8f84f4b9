// Internal launch interfaces between capi.cu and the kernel translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace f3r {

// 1: launch the hot-chain kernels with programmatic stream serialization (PDL); F3R_PDL=0 / f3r_set_option("pdl", 0) disable
extern int g_pdl;
bool pdl_enabled();
// fills `attr` (room for 2) with the cluster dimension (if cluster > 1) and the PDL attribute (if enabled); returns the count
int launch_attrs(cudaLaunchAttribute* attr, int cluster);

enum { EPI_STORE = 0, EPI_ROPE = 1, EPI_IDXEMB = 2, EPI_CONVT = 3, EPI_FINAL = 4 };
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_GELU = 2 };

struct GemmArgs {
  int M, N, K, taps;
  int W, H, NB, bw, bh, tiles_x, tiles_y;
  int bw_log2;  // bw is a power of two
  int num_m_tiles, num_n_tiles;
  int epi, act, out0_f32, res0_f32;
  int ldo;               // row stride (elements) of out0 / out1 / res0 / res1
  int split_col, ldo_b;  // columns >= split_col go to out0b (row stride ldo_b); 0 = no split
  int tok_per_img, grid_w, rope_cols;  // EPI_ROPE / EPI_IDXEMB
  int ct_k, ct_cout;                   // EPI_CONVT
  int tma_epi;                         // 0: generic epilogue, 1: TMA store of out0(/out0b), 2: TMA reduce-add into fp32 out0
  int sbx_log2;                        // TMA-store box = (32 ch, sbx, 32/sbx) pixels, sbx = min(bw, 32)
  int k_split;                         // K slices per output tile (>1 only with tma_epi == 2: partial sums reduce-added)
  int debug;                           // F3R_GEMM_DEBUG bitmask (1: no epilogue stores) - timing experiments only
  const float* bias;
  const void* res0;
  const void* res1;
  void* out0;
  void* out0b;
  void* out1;
  const float* rope_cos;
  const float* rope_sin;
  const float* emb_table;
  const int* emb_ids;
  const float* w4;
  const float* b4;
  float* pts;
  float* conf;
};

cudaError_t launch_gemm(int block_n, int cluster, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to0,
                        const CUtensorMap& to0b, const GemmArgs& a, int num_sms, cudaStream_t stream);

struct AttnArgs {
  int batch, heads, sq, skv;  // per-batch query / key lengths
  int q_tiles;                // ceil(sq / 256)
  float scale_log2;           // softmax scale * log2(e)
  int ldo;                    // row stride of out (elements)
  void* out;                  // bf16 [batch*sq, ldo], head h at columns h*64
  float* lse;                 // optional fp32 [batch, heads, sq] log-sum-exp (natural log)
  // key range of this launch inside the kv buffer: rows [kv_row0, kv_row0 + skv) of every batch
  int kv_row0;
  // key-slice partials: the key blocks are cut into n_split slices (one CTA each per query tile); with part_o != NULL
  // slice s writes its normalised fp32 output / LSE into slot part_base + s (merged by launch_attention_merge)
  int n_split;
  int part_base;
  float* part_o;              // fp32 [slots, batch*sq, heads*64]
  float* part_lse;            // fp32 [slots, batch, heads, sq]
};
cudaError_t launch_attention_merge(const float* part_o, const float* part_lse, int n_parts, int batch, int heads, int sq,
                                   void* out, int ldo, cudaStream_t stream);
cudaError_t launch_attention(const CUtensorMap& tq, const CUtensorMap& tkv, const AttnArgs& a, cudaStream_t stream);
extern int g_attn_emu;    // exponential pairs (of every 8) evaluated on the FMA pipe, -1 = default
extern int g_attn_split;  // softmax threads per query row (1 or 2), -1 = default

// parity mode (attention_x3.cu): hi/lo-split bf16 operands, fp32 out (AttnArgs.out is float*, q_tiles = ceil(sq / 128))
cudaError_t launch_attention_x3(const CUtensorMap& tq3, const CUtensorMap& tk3, const CUtensorMap& tv2,
                                const AttnArgs& a, cudaStream_t stream);
cudaError_t launch_attn_split(const float* q, int ldq, const float* kv, int ldkv, void* q3, void* k3, void* v2,
                              size_t rows_q, size_t rows_kv, int heads, cudaStream_t stream);
cudaError_t launch_split3(const float* in, void* out, size_t rows, int k, int relu, cudaStream_t stream);
cudaError_t launch_add_f32(float* dst, const float* src, size_t n, cudaStream_t stream);

cudaError_t launch_layernorm(const float* x, const float* w, const float* b, void* out, int out_f32, int rows,
                             int dim, float eps, cudaStream_t stream);
cudaError_t launch_im2col_patch(const float* img, void* out, int out_f32, int n, int H, int W, int patch,
                                cudaStream_t stream);
cudaError_t launch_im2col3x3s2(const void* in, void* out, int n, int H, int W, int C, int Ho, int Wo,
                               cudaStream_t stream);
cudaError_t launch_upsample2x(const void* in, void* out, int f32, int n, int H, int W, int C, int Ho, int Wo,
                              int Hfull, int Wfull, cudaStream_t stream);
cudaError_t launch_cast_bf16(const float* in, void* out, size_t n, cudaStream_t stream);

// image ingest (ingest.cu)
int resample_ksize(int in_size, int out_size, int filter);
int resample_coeffs(int in_size, int out_size, int filter, int32_t* bounds, int32_t* kk);
cudaError_t launch_ingest(const uint8_t* src, int h, int w, int oh, int ow, const int32_t* hb, const int32_t* hk, int hks,
                          int h_span_max, const int32_t* vb, const int32_t* vk, int vks, uint8_t* tmp, int left, int top,
                          int cw, int ch, float* out, cudaStream_t stream);

// geometry tail (geometry.cu)
cudaError_t launch_conf_quantile(const float* conf, int views, int n, float q, float* thr, cudaStream_t stream);
size_t similarity_fit_workspace(int views);
cudaError_t launch_similarity_fit(const float* x, const float* y, const float* conf, const float* thr,
                                  const uint8_t* valid, int views, int n, float* rts, double* workspace,
                                  cudaStream_t stream);
cudaError_t launch_similarity_apply(const float* x, const float* rts, float* out, int views, int n, cudaStream_t stream);
size_t focal_workspace(int views);
cudaError_t launch_focal_weiszfeld(const float* pts, const float* conf, const float* thr, const float* pp, int views,
                                   int H, int W, int iters, float* focal, double* workspace, cudaStream_t stream);

// camera poses (pnp.cu): 4 launches, then PNP_LM_STEPS + 1 refit passes of 2 launches
constexpr int PNP_LM_STEPS = 10;
size_t pnp_workspace(int views, int n, int hyps);
cudaError_t launch_pnp_ransac(const float* pts, const uint8_t* mask, int views, int H, int W, const float* focals,
                              int n_focals, const float* pp, int iters, int32_t* scores, int32_t* best, double* c2w,
                              void* workspace, cudaStream_t stream);

}  // namespace f3r
