// extern "C" boundary of libfast3r_b200.so (see include/fast3r_b200.h).  Builds the TMA descriptors
// (cuTensorMapEncodeTiled through cudaGetDriverEntryPoint, so libcuda is not a link-time dependency),
// validates arguments and enqueues the kernels on the caller's stream.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/fast3r_b200.h"
#include "f3r_kernels.h"

namespace {

thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};

int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}
int check(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  return fail("%s: %s", what, cudaGetErrorString(e));
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// Tensor map with zero OOB fill.  dims[0] is the contiguous dimension.  Defaults: bf16, 128B swizzle (MMA operands).
int make_tmap(CUtensorMap* m, const void* ptr, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
              const uint32_t* box, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
              CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return fail("cuTensorMapEncodeTiled not available (no CUDA driver?)");
  cuuint64_t gd[5];
  cuuint64_t gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i < rank - 1; ++i) gs[i] = strides_bytes[i];
  if (reinterpret_cast<uintptr_t>(ptr) & 15) return fail("tensor map base not 16-byte aligned");
  for (int i = 0; i < rank - 1; ++i)
    if (gs[i] % 16) return fail("tensor map stride %d (%llu B) not a multiple of 16", i, (unsigned long long)gs[i]);
  CUresult r = enc(m, dtype, rank, const_cast<void*>(ptr), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d", static_cast<int>(r));
  return 0;
}

int num_sms() {
  static int cache[64] = {0};  // per device: one process may drive several GPUs
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int& n = cache[dev & 63];
  if (n) return n;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  return n;
}

}  // namespace

extern "C" {

const char* f3r_last_error(void) { return g_err; }
int f3r_abi_version(void) { return F3R_ABI_VERSION; }
size_t f3r_gemm_desc_size(void) { return sizeof(f3r_gemm_desc); }
uint64_t f3r_launch_count(void) { return g_launches.load(); }

int f3r_set_option(const char* name, int32_t value) {
  if (!name) return fail("f3r_set_option: null name");
  if (!strcmp(name, "attn_emu")) {
    if (value < -1 || value > 3) return fail("f3r_set_option: attn_emu must be in [-1, 3]");
    f3r::g_attn_emu = value;
    return 0;
  }
  if (!strcmp(name, "pdl")) {
    if (value != 0 && value != 1) return fail("f3r_set_option: pdl must be 0 or 1");
    f3r::g_pdl = value;
    return 0;
  }
  if (!strcmp(name, "attn_split")) {
    if (value != -1 && value != 1 && value != 2) return fail("f3r_set_option: attn_split must be -1, 1 or 2");
    f3r::g_attn_split = value;
    return 0;
  }
  return fail("f3r_set_option: unknown option '%s'", name);
}

int f3r_gemm(const f3r_gemm_desc* d, void* stream) {
  if (!d || !d->a || !d->wt) return fail("f3r_gemm: null operand");
  if (d->n <= 0 || d->k <= 0 || d->w <= 0 || d->h <= 0 || d->nb <= 0) return fail("f3r_gemm: bad shape");
  if (d->n % 32) return fail("f3r_gemm: n=%d must be a multiple of 32", d->n);
  if (d->k % 8 || d->a_ld % 8) return fail("f3r_gemm: k=%d and a_ld=%d must be multiples of 8", d->k, d->a_ld);
  if (d->taps != 1 && d->taps != 9) return fail("f3r_gemm: taps must be 1 or 9");
  if (d->epi == F3R_EPI_FINAL && d->n != 128) return fail("f3r_gemm: FINAL epilogue needs n == 128");
  if (d->epi == F3R_EPI_CONVT && (d->ct_k <= 0 || d->ct_cout % 32 || d->n != d->ct_k * d->ct_k * d->ct_cout))
    return fail("f3r_gemm: bad CONVT geometry");
  if (d->epi == F3R_EPI_ROPE && (!d->rope_cos || !d->rope_sin || d->tok_per_img <= 0 || d->grid_w <= 0))
    return fail("f3r_gemm: bad ROPE arguments");
  if (d->epi == F3R_EPI_IDXEMB && (!d->emb_table || !d->emb_ids || d->tok_per_img < 0))
    return fail("f3r_gemm: bad IDXEMB arguments");

  f3r::GemmArgs a;
  memset(&a, 0, sizeof(a));
  a.M = d->w * d->h * d->nb; a.N = d->n; a.K = d->k; a.taps = d->taps;
  a.W = d->w; a.H = d->h; a.NB = d->nb;
  // pixel tile (bw x bh = 128) minimising the number of tiles
  int best_bw = 128; long best_tiles = -1;
  for (int bw = 128; bw >= 1; bw >>= 1) {
    const int bh = 128 / bw;
    const long tiles = static_cast<long>((d->w + bw - 1) / bw) * ((d->h + bh - 1) / bh);
    if (best_tiles < 0 || tiles < best_tiles) { best_tiles = tiles; best_bw = bw; }
  }
  a.bw = best_bw; a.bh = 128 / best_bw;
  a.bw_log2 = 0;
  while ((1 << a.bw_log2) < a.bw) ++a.bw_log2;
  a.sbx_log2 = a.bw_log2 < 5 ? a.bw_log2 : 5;
  a.tiles_x = (d->w + a.bw - 1) / a.bw; a.tiles_y = (d->h + a.bh - 1) / a.bh;
  a.num_m_tiles = a.tiles_x * a.tiles_y * d->nb;
  int block_n = 128;
  if (d->epi != F3R_EPI_FINAL && d->n > 128) {
    const long tiles256 = static_cast<long>(a.num_m_tiles) * ((d->n + 255) / 256);
    if (tiles256 >= num_sms()) block_n = 256;
  }
  a.num_n_tiles = (d->n + block_n - 1) / block_n;
  // CTA pairs sharing the weight tile through TMA multicast (F3R_GEMM_CLUSTER=1 disables, for A/B measurements)
  static int cluster_pref = -1;
  if (cluster_pref < 0) {
    const char* e = getenv("F3R_GEMM_CLUSTER");
    cluster_pref = (e && e[0] == '1') ? 1 : 2;
  }
  const int cluster = (cluster_pref == 2 && a.num_m_tiles >= 2) ? 2 : 1;
  static int dbg = -1, tma_pref = -1;
  if (dbg < 0) { const char* e = getenv("F3R_GEMM_DEBUG"); dbg = e ? atoi(e) : 0; }
  if (tma_pref < 0) { const char* e = getenv("F3R_GEMM_TMA_EPI"); tma_pref = (e && e[0] == '0') ? 0 : 1; }
  a.debug = dbg;
  a.epi = d->epi; a.act = d->act; a.out0_f32 = d->out0_f32; a.res0_f32 = d->res0_f32;
  a.ldo = d->ldo > 0 ? d->ldo : d->n;
  a.split_col = d->split_col; a.ldo_b = d->ldo_b;
  a.tok_per_img = d->tok_per_img; a.grid_w = d->grid_w; a.rope_cols = d->rope_cols;
  a.ct_k = d->ct_k; a.ct_cout = d->ct_cout;
  a.bias = d->bias; a.res0 = d->res0; a.res1 = d->res1;
  a.out0 = d->out0; a.out0b = d->out0b; a.out1 = d->out1;
  a.rope_cos = d->rope_cos; a.rope_sin = d->rope_sin;
  a.emb_table = d->emb_table; a.emb_ids = d->emb_ids;
  a.w4 = d->w4; a.b4 = d->b4; a.pts = d->pts; a.conf = d->conf;
  if (a.split_col && (a.split_col % 32 || !a.out0b)) return fail("f3r_gemm: bad column split");

  CUtensorMap ta, tb;
  {
    const uint64_t ld = static_cast<uint64_t>(d->a_ld) * 2;
    const uint64_t dims[4] = {static_cast<uint64_t>(d->k), static_cast<uint64_t>(d->w),
                              static_cast<uint64_t>(d->h), static_cast<uint64_t>(d->nb)};
    const uint64_t str[3] = {ld, ld * d->w, ld * d->w * d->h};
    const uint32_t box[4] = {64, static_cast<uint32_t>(a.bw), static_cast<uint32_t>(a.bh), 1};
    if (make_tmap(&ta, d->a, 4, dims, str, box)) return 1;
  }
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(d->k), static_cast<uint64_t>(d->taps),
                              static_cast<uint64_t>(d->n)};
    const uint64_t str[2] = {static_cast<uint64_t>(d->k) * 2, static_cast<uint64_t>(d->k) * 2 * d->taps};
    const uint32_t box[3] = {64, 1, static_cast<uint32_t>(block_n / cluster)};
    if (make_tmap(&tb, d->wt, 3, dims, str, box)) return 1;
  }
  // TMA epilogue for the hot cases: plain (activated) stores, and the in-place fp32 residual update as a reduce-add
  CUtensorMap to0, to0b;
  memset(&to0, 0, sizeof(to0));
  memset(&to0b, 0, sizeof(to0b));
  const bool plain = (d->epi == F3R_EPI_STORE || d->epi == F3R_EPI_ROPE || d->epi == F3R_EPI_IDXEMB) && d->out0 &&
                     !d->out1 && !d->res1;
  if (tma_pref && plain && !d->res0) a.tma_epi = 1;
  else if (tma_pref && plain && d->res0 == d->out0 && d->res0_f32 && d->out0_f32 && !d->split_col) a.tma_epi = 2;
  if (a.tma_epi) {
    const uint64_t es = d->out0_f32 ? 4 : 2;
    const CUtensorMapDataType dt = d->out0_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    const CUtensorMapSwizzle sw = d->out0_f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const uint32_t sbx = 1u << a.sbx_log2;
    const uint32_t box[4] = {32, sbx, 32 / sbx, 1};
    const uint64_t ncols0 = a.split_col ? a.split_col : d->n;
    {
      const uint64_t ld = static_cast<uint64_t>(a.ldo) * es;
      const uint64_t dims[4] = {ncols0, static_cast<uint64_t>(d->w), static_cast<uint64_t>(d->h),
                                static_cast<uint64_t>(d->nb)};
      const uint64_t str[3] = {ld, ld * d->w, ld * d->w * d->h};
      if (make_tmap(&to0, d->out0, 4, dims, str, box, dt, sw)) return 1;
    }
    if (a.split_col) {
      const uint64_t ld = static_cast<uint64_t>(a.ldo_b) * es;
      const uint64_t dims[4] = {static_cast<uint64_t>(d->n - a.split_col), static_cast<uint64_t>(d->w),
                                static_cast<uint64_t>(d->h), static_cast<uint64_t>(d->nb)};
      const uint64_t str[3] = {ld, ld * d->w, ld * d->w * d->h};
      if (make_tmap(&to0b, d->out0b, 4, dims, str, box, dt, sw)) return 1;
    }
  }
  a.k_split = 1;
  static int ksplit_pref = -1;  // F3R_GEMM_KSPLIT=1 disables the K slicing (A/B measurements)
  if (ksplit_pref < 0) { const char* e = getenv("F3R_GEMM_KSPLIT"); ksplit_pref = (e && e[0] == '1') ? 1 : 0; }
  if (a.tma_epi == 2 && d->taps == 1 && ksplit_pref != 1) {
    // x += A W^T with fewer output tiles than SM (pairs): cut K into slices, each CTA reduce-adds its partial sum
    const long slots = num_sms() / cluster;
    const long items = static_cast<long>((a.num_m_tiles + cluster - 1) / cluster) * a.num_n_tiles;
    const int k_iters = (d->k + 63) / 64;
    double best = 1e30;
    for (int s = 1; s <= 4 && (s == 1 || k_iters / s >= 16); ++s) {  // (short K: the reduce-add epilogue dominates, slicing loses)
      const double cost = static_cast<double>((items * s + slots - 1) / slots) / s * (1.0 + 0.03 * (s - 1));
      if (cost < best - 1e-9) { best = cost; a.k_split = s; }
    }
  }
  g_launches++;
  return check(f3r::launch_gemm(block_n, cluster, ta, tb, to0, to0b, a, num_sms(), static_cast<cudaStream_t>(stream)),
               "f3r_gemm");
}

static int attention_impl(const char* what, const void* q, int32_t ldq, const void* kv, int32_t ldkv,
                          int32_t kv_rows_total, int32_t kv_row0, void* out, int32_t ldo, float* lse, float* part_o,
                          float* part_lse, int32_t part_base, int32_t n_split, int32_t batch, int32_t heads, int32_t sq,
                          int32_t skv, float scale, void* stream) {
  if (!q || !kv) return fail("%s: null operand", what);
  if (batch <= 0 || heads <= 0 || sq <= 0 || skv <= 0) return fail("%s: bad shape", what);
  if (ldq % 8 || ldkv % 8 || ldq < heads * 64 || ldkv < 2 * heads * 64) return fail("%s: bad leading dimensions", what);
  if (kv_row0 < 0 || kv_row0 + skv > kv_rows_total) return fail("%s: key range outside the kv buffer", what);
  if (n_split < 1 || n_split > (skv + 127) / 128) return fail("%s: n_split=%d must be in [1, #key blocks]", what, n_split);
  CUtensorMap tq, tkv;
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(heads) * 64, static_cast<uint64_t>(sq),
                              static_cast<uint64_t>(batch)};
    const uint64_t str[2] = {static_cast<uint64_t>(ldq) * 2, static_cast<uint64_t>(ldq) * 2 * sq};
    const uint32_t box[3] = {64, 128, 1};
    if (make_tmap(&tq, q, 3, dims, str, box)) return 1;
  }
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(heads) * 128, static_cast<uint64_t>(kv_rows_total),
                              static_cast<uint64_t>(batch)};
    const uint64_t str[2] = {static_cast<uint64_t>(ldkv) * 2, static_cast<uint64_t>(ldkv) * 2 * kv_rows_total};
    const uint32_t box[3] = {64, 128, 1};
    if (make_tmap(&tkv, kv, 3, dims, str, box)) return 1;
  }
  f3r::AttnArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = batch; a.heads = heads; a.sq = sq; a.skv = skv;
  a.q_tiles = (sq + 255) / 256;
  a.scale_log2 = scale * 1.4426950408889634f;
  a.ldo = ldo; a.out = out; a.lse = lse;
  a.kv_row0 = kv_row0; a.n_split = n_split; a.part_base = part_base; a.part_o = part_o; a.part_lse = part_lse;
  g_launches++;
  return check(f3r::launch_attention(tq, tkv, a, static_cast<cudaStream_t>(stream)), what);
}

int f3r_attention(const void* q, int32_t ldq, const void* kv, int32_t ldkv, void* out, int32_t ldo, float* lse,
                  int32_t batch, int32_t heads, int32_t sq, int32_t skv, float scale, void* stream) {
  if (!out) return fail("f3r_attention: null operand");
  if (ldo % 8 || ldo < heads * 64) return fail("f3r_attention: bad leading dimensions");
  return attention_impl("f3r_attention", q, ldq, kv, ldkv, skv, 0, out, ldo, lse, nullptr, nullptr, 0, 1, batch, heads,
                        sq, skv, scale, stream);
}

int f3r_attention_partial(const void* q, int32_t ldq, const void* kv, int32_t ldkv, int32_t kv_rows_total,
                          int32_t kv_row0, int32_t skv, int32_t n_split, float* part_o, float* part_lse,
                          int32_t part_base, int32_t batch, int32_t heads, int32_t sq, float scale, void* stream) {
  if (!part_o || !part_lse || part_base < 0) return fail("f3r_attention_partial: bad partial buffers");
  return attention_impl("f3r_attention_partial", q, ldq, kv, ldkv, kv_rows_total, kv_row0, nullptr, 0, nullptr, part_o,
                        part_lse, part_base, n_split, batch, heads, sq, skv, scale, stream);
}

int f3r_attention_merge(const float* part_o, const float* part_lse, int32_t n_parts, void* out, int32_t ldo,
                        int32_t batch, int32_t heads, int32_t sq, void* stream) {
  if (!part_o || !part_lse || !out || n_parts < 1) return fail("f3r_attention_merge: bad arguments");
  if (ldo % 8 || ldo < heads * 64) return fail("f3r_attention_merge: bad leading dimension");
  g_launches++;
  return check(f3r::launch_attention_merge(part_o, part_lse, n_parts, batch, heads, sq, out, ldo,
                                           static_cast<cudaStream_t>(stream)), "f3r_attention_merge");
}

int f3r_layernorm(const float* x, const float* w, const float* b, void* out, int32_t out_f32, int32_t rows,
                  int32_t dim, float eps, void* stream) {
  if (!x || !w || !b || !out) return fail("f3r_layernorm: null operand");
  g_launches++;
  return check(f3r::launch_layernorm(x, w, b, out, out_f32, rows, dim, eps, static_cast<cudaStream_t>(stream)),
               "f3r_layernorm (dim must be one of 128,256,384,512,768,1024)");
}

int f3r_im2col_patch(const float* img, void* out, int32_t out_f32, int32_t n, int32_t h, int32_t w, void* stream) {
  if (!img || !out) return fail("f3r_im2col_patch: null operand");
  g_launches++;
  return check(f3r::launch_im2col_patch(img, out, out_f32, n, h, w, 16, static_cast<cudaStream_t>(stream)),
               "f3r_im2col_patch");
}

int f3r_im2col3x3s2(const void* in, void* out, int32_t n, int32_t h, int32_t w, int32_t c, int32_t ho, int32_t wo,
                    void* stream) {
  if (!in || !out) return fail("f3r_im2col3x3s2: null operand");
  g_launches++;
  return check(f3r::launch_im2col3x3s2(in, out, n, h, w, c, ho, wo, static_cast<cudaStream_t>(stream)),
               "f3r_im2col3x3s2");
}

int f3r_upsample2x(const void* in, void* out, int32_t f32, int32_t n, int32_t h, int32_t w, int32_t c, int32_t ho,
                   int32_t wo, void* stream) {
  if (!in || !out) return fail("f3r_upsample2x: null operand");
  if (ho > 2 * h || wo > 2 * w) return fail("f3r_upsample2x: window larger than the x2 output");
  g_launches++;
  return check(f3r::launch_upsample2x(in, out, f32, n, h, w, c, ho, wo, 2 * h, 2 * w,
                                      static_cast<cudaStream_t>(stream)),
               "f3r_upsample2x");
}

int f3r_split3(const float* in, void* out, size_t rows, int32_t k, int32_t relu, void* stream) {
  if (!in || !out) return fail("f3r_split3: null operand");
  if (k <= 0 || k % 8) return fail("f3r_split3: k=%d must be a positive multiple of 8", k);
  g_launches++;
  return check(f3r::launch_split3(in, out, rows, k, relu, static_cast<cudaStream_t>(stream)), "f3r_split3");
}

int f3r_add_f32(float* dst, const float* src, size_t count, void* stream) {
  if (!dst || !src) return fail("f3r_add_f32: null operand");
  g_launches++;
  return check(f3r::launch_add_f32(dst, src, count, static_cast<cudaStream_t>(stream)), "f3r_add_f32");
}

size_t f3r_attention_x3_workspace(int32_t batch, int32_t heads, int32_t sq, int32_t skv) {
  // q3 [batch*sq, heads*192] + k3 [batch*skv, heads*192] + v2 [batch*skv, heads*128] bf16, each 256-byte aligned
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  return al(static_cast<size_t>(batch) * sq * heads * 192 * 2) + al(static_cast<size_t>(batch) * skv * heads * 192 * 2) +
         al(static_cast<size_t>(batch) * skv * heads * 128 * 2);
}

int f3r_attention_x3(const float* q, int32_t ldq, const float* kv, int32_t ldkv, float* out, int32_t ldo, float* lse,
                     void* workspace, size_t workspace_bytes, int32_t batch, int32_t heads, int32_t sq, int32_t skv,
                     float scale, void* stream) {
  if (!q || !kv || !out || !workspace) return fail("f3r_attention_x3: null operand");
  if (batch <= 0 || heads <= 0 || sq <= 0 || skv <= 0) return fail("f3r_attention_x3: bad shape");
  if (ldq % 4 || ldkv % 4 || ldo % 4 || ldq < heads * 64 || ldkv < 2 * heads * 64 || ldo < heads * 64)
    return fail("f3r_attention_x3: bad leading dimensions");
  if (workspace_bytes < f3r_attention_x3_workspace(batch, heads, sq, skv))
    return fail("f3r_attention_x3: workspace too small (%zu < %zu bytes)", workspace_bytes,
                f3r_attention_x3_workspace(batch, heads, sq, skv));
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail("f3r_attention_x3: workspace not 256-byte aligned");
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  uint8_t* w = static_cast<uint8_t*>(workspace);
  void* q3 = w;
  void* k3 = w + al(static_cast<size_t>(batch) * sq * heads * 192 * 2);
  void* v2 = static_cast<uint8_t*>(k3) + al(static_cast<size_t>(batch) * skv * heads * 192 * 2);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  g_launches++;
  if (check(f3r::launch_attn_split(q, ldq, kv, ldkv, q3, k3, v2, static_cast<size_t>(batch) * sq,
                                   static_cast<size_t>(batch) * skv, heads, st), "f3r_attention_x3 (split)"))
    return 1;
  CUtensorMap tq3, tk3, tv2;
  const uint32_t box[3] = {64, 128, 1};
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(heads) * 192, static_cast<uint64_t>(sq), static_cast<uint64_t>(batch)};
    const uint64_t str[2] = {static_cast<uint64_t>(heads) * 192 * 2, static_cast<uint64_t>(heads) * 192 * 2 * sq};
    if (make_tmap(&tq3, q3, 3, dims, str, box)) return 1;
  }
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(heads) * 192, static_cast<uint64_t>(skv), static_cast<uint64_t>(batch)};
    const uint64_t str[2] = {static_cast<uint64_t>(heads) * 192 * 2, static_cast<uint64_t>(heads) * 192 * 2 * skv};
    if (make_tmap(&tk3, k3, 3, dims, str, box)) return 1;
  }
  {
    const uint64_t dims[3] = {static_cast<uint64_t>(heads) * 128, static_cast<uint64_t>(skv), static_cast<uint64_t>(batch)};
    const uint64_t str[2] = {static_cast<uint64_t>(heads) * 128 * 2, static_cast<uint64_t>(heads) * 128 * 2 * skv};
    if (make_tmap(&tv2, v2, 3, dims, str, box)) return 1;
  }
  f3r::AttnArgs a;
  memset(&a, 0, sizeof(a));
  a.batch = batch; a.heads = heads; a.sq = sq; a.skv = skv;
  a.q_tiles = (sq + 127) / 128;
  a.scale_log2 = scale * 1.4426950408889634f;
  a.ldo = ldo; a.out = out; a.lse = lse;
  g_launches++;
  return check(f3r::launch_attention_x3(tq3, tk3, tv2, a, st), "f3r_attention_x3");
}

int f3r_resample_ksize(int32_t in_size, int32_t out_size, int32_t filter) {
  if (in_size <= 0 || out_size <= 0 || (filter != 0 && filter != 1)) return -1;
  return f3r::resample_ksize(in_size, out_size, filter);
}

int f3r_resample_coeffs(int32_t in_size, int32_t out_size, int32_t filter, int32_t* bounds, int32_t* kk) {
  if (in_size <= 0 || out_size <= 0 || (filter != 0 && filter != 1) || !bounds || !kk) {
    fail("f3r_resample_coeffs: bad arguments");
    return -1;
  }
  return f3r::resample_coeffs(in_size, out_size, filter, bounds, kk);
}

int f3r_ingest_rgb8(const uint8_t* src, int32_t h, int32_t w, int32_t oh, int32_t ow, const int32_t* hb, const int32_t* hk,
                    int32_t hks, int32_t h_span_max, const int32_t* vb, const int32_t* vk, int32_t vks, uint8_t* tmp,
                    int32_t left, int32_t top, int32_t cw, int32_t ch, float* out, void* stream) {
  if (!src || !out) return fail("f3r_ingest_rgb8: null operand");
  if (h <= 0 || w <= 0 || oh <= 0 || ow <= 0 || cw <= 0 || ch <= 0) return fail("f3r_ingest_rgb8: bad shape");
  if (left < 0 || top < 0 || left + cw > ow || top + ch > oh) return fail("f3r_ingest_rgb8: crop box outside the resized image");
  if ((ow != w) != (hk != nullptr) || (oh != h) != (vk != nullptr))
    return fail("f3r_ingest_rgb8: tap tables must be given exactly for the resized dimensions");
  if (hk && (!hb || !tmp || hks <= 0 || h_span_max <= 0)) return fail("f3r_ingest_rgb8: incomplete horizontal pass arguments");
  if (vk && (!vb || vks <= 0)) return fail("f3r_ingest_rgb8: incomplete vertical pass arguments");
  g_launches += hk ? 2 : 1;
  return check(f3r::launch_ingest(src, h, w, oh, ow, hb, hk, hks, h_span_max, vb, vk, vks, tmp, left, top, cw, ch, out,
                                  static_cast<cudaStream_t>(stream)), "f3r_ingest_rgb8");
}

// ---------------------------------------------------------------- geometry tail
int f3r_conf_quantile(const float* conf, int32_t views, int32_t n, float q, float* thr, void* stream) {
  if (!conf || !thr) return fail("f3r_conf_quantile: null operand");
  if (views <= 0 || n <= 0 || n > (1 << 24)) return fail("f3r_conf_quantile: bad shape (n must be in [1, 2^24]: ranks are fp32)");
  if (!(q >= 0.f && q <= 1.f)) return fail("f3r_conf_quantile: q must be in [0, 1]");
  g_launches++;
  return check(f3r::launch_conf_quantile(conf, views, n, q, thr, static_cast<cudaStream_t>(stream)), "f3r_conf_quantile");
}

size_t f3r_similarity_fit_workspace(int32_t views) { return views > 0 ? f3r::similarity_fit_workspace(views) : 0; }

int f3r_similarity_fit(const float* x, const float* y, const float* conf, const float* thr, const uint8_t* valid,
                       int32_t views, int32_t n, float* rts, void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !y || !rts || !workspace) return fail("f3r_similarity_fit: null operand");
  if (views <= 0 || views > 65535 || n <= 0 || n > (1 << 29)) return fail("f3r_similarity_fit: bad shape");
  if ((conf != nullptr) != (thr != nullptr)) return fail("f3r_similarity_fit: conf and thr must be given together");
  if (workspace_bytes < f3r::similarity_fit_workspace(views)) return fail("f3r_similarity_fit: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace) & 7) return fail("f3r_similarity_fit: workspace not 8-byte aligned");
  g_launches += conf ? 4 : 2;
  return check(f3r::launch_similarity_fit(x, y, conf, thr, valid, views, n, rts, static_cast<double*>(workspace),
                                          static_cast<cudaStream_t>(stream)), "f3r_similarity_fit");
}

int f3r_similarity_apply(const float* x, const float* rts, float* out, int32_t views, int32_t n, void* stream) {
  if (!x || !rts || !out) return fail("f3r_similarity_apply: null operand");
  if (views <= 0 || views > 65535 || n <= 0 || n > (1 << 29)) return fail("f3r_similarity_apply: bad shape");
  g_launches++;
  return check(f3r::launch_similarity_apply(x, rts, out, views, n, static_cast<cudaStream_t>(stream)), "f3r_similarity_apply");
}

size_t f3r_focal_workspace(int32_t views) { return views > 0 ? f3r::focal_workspace(views) : 0; }

int f3r_focal_weiszfeld(const float* pts, const float* conf, const float* thr, const float* pp, int32_t views, int32_t h,
                        int32_t w, int32_t iters, float* focal, void* workspace, size_t workspace_bytes, void* stream) {
  if (!pts || !focal || !workspace) return fail("f3r_focal_weiszfeld: null operand");
  if (views <= 0 || views > 65535 || h <= 0 || w <= 0 || static_cast<int64_t>(h) * w > (1 << 29))
    return fail("f3r_focal_weiszfeld: bad shape");
  if (iters < 0 || iters > 10000) return fail("f3r_focal_weiszfeld: bad iteration count");
  if ((conf != nullptr) != (thr != nullptr)) return fail("f3r_focal_weiszfeld: conf and thr must be given together");
  if (workspace_bytes < f3r::focal_workspace(views)) return fail("f3r_focal_weiszfeld: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace) & 7) return fail("f3r_focal_weiszfeld: workspace not 8-byte aligned");
  g_launches += static_cast<uint64_t>(iters) + 2;
  return check(f3r::launch_focal_weiszfeld(pts, conf, thr, pp, views, h, w, iters, focal, static_cast<double*>(workspace),
                                           static_cast<cudaStream_t>(stream)), "f3r_focal_weiszfeld");
}

// ---------------------------------------------------------------- camera poses
static bool pnp_shape_ok(int32_t views, int32_t h, int32_t w, int32_t n_focals, int32_t iters) {
  return views > 0 && views <= 65535 && h > 0 && w > 0 && static_cast<int64_t>(h) * w <= (1 << 24) && n_focals > 0 &&
         iters > 0 && static_cast<int64_t>(n_focals) * iters <= (1 << 20);
}

size_t f3r_pnp_workspace(int32_t views, int32_t h, int32_t w, int32_t n_focals, int32_t iters) {
  return pnp_shape_ok(views, h, w, n_focals, iters) ? f3r::pnp_workspace(views, h * w, n_focals * iters) : 0;
}

int f3r_pnp_ransac(const float* pts, const uint8_t* mask, int32_t views, int32_t h, int32_t w, const float* focals,
                   int32_t n_focals, const float* pp, int32_t iters, int32_t* scores, int32_t* best, double* c2w,
                   void* workspace, size_t workspace_bytes, void* stream) {
  if (!pts || !mask || !focals || !scores || !best || !c2w || !workspace) return fail("f3r_pnp_ransac: null operand");
  if (n_focals < 1) return fail("f3r_pnp_ransac: n_focals must be >= 1");
  if (iters < 1) return fail("f3r_pnp_ransac: iters must be >= 1");
  if (!pnp_shape_ok(views, h, w, n_focals, iters))
    return fail("f3r_pnp_ransac: bad shape (views <= 65535, h*w <= 2^24, n_focals*iters <= 2^20)");
  if (workspace_bytes < f3r::pnp_workspace(views, h * w, n_focals * iters))
    return fail("f3r_pnp_ransac: workspace too small (%zu < %zu bytes)", workspace_bytes,
                f3r::pnp_workspace(views, h * w, n_focals * iters));
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail("f3r_pnp_ransac: workspace not 256-byte aligned");
  g_launches += 4 + 2 * (f3r::PNP_LM_STEPS + 1);
  return check(f3r::launch_pnp_ransac(pts, mask, views, h, w, focals, n_focals, pp, iters, scores, best, c2w, workspace,
                                      static_cast<cudaStream_t>(stream)), "f3r_pnp_ransac");
}

// ---------------------------------------------------------------- block-level entry points
size_t f3r_transformer_workspace(int32_t rows, int32_t dim, int32_t hidden) {
  // h [rows, dim] | q [rows, dim] | kv [rows, 2 dim] | att [rows, dim] | hid [rows, hidden], bf16, 256-byte aligned parts
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  const size_t r = static_cast<size_t>(rows);
  return 3 * al(r * dim * 2) + al(r * 2 * dim * 2) + al(r * hidden * 2);
}

int f3r_transformer_blocks(const f3r_block_weights* blocks, int32_t n_blocks, float* x, int32_t batch, int32_t seq,
                           int32_t dim, int32_t heads, int32_t hidden, float eps, float scale, int32_t rope_grid_w,
                           int32_t rope_tok_per_img, const float* rope_cos, const float* rope_sin, void* workspace,
                           size_t workspace_bytes, void* stream) {
  if (!blocks || n_blocks <= 0 || !x || !workspace) return fail("f3r_transformer_blocks: null operand");
  if (batch <= 0 || seq <= 0 || dim != heads * 64 || hidden <= 0) return fail("f3r_transformer_blocks: bad shape (head_dim must be 64)");
  const int32_t rows = batch * seq;
  if (workspace_bytes < f3r_transformer_workspace(rows, dim, hidden)) return fail("f3r_transformer_blocks: workspace too small");
  if (reinterpret_cast<uintptr_t>(workspace) & 255) return fail("f3r_transformer_blocks: workspace not 256-byte aligned");
  auto al = [](size_t b) { return (b + 255) & ~static_cast<size_t>(255); };
  uint8_t* w = static_cast<uint8_t*>(workspace);
  const size_t r = static_cast<size_t>(rows);
  void* h = w;
  void* q = w + al(r * dim * 2);
  void* kv = static_cast<uint8_t*>(q) + al(r * dim * 2);
  void* att = static_cast<uint8_t*>(kv) + al(r * 2 * dim * 2);
  void* hid = static_cast<uint8_t*>(att) + al(r * dim * 2);
  const bool rope = rope_cos != nullptr;
  for (int i = 0; i < n_blocks; ++i) {
    const f3r_block_weights& b = blocks[i];
    // x += proj(attention(rope(q), rope(k), v));  x += fc2(gelu(fc1(LN(x))))     (fast3r/croco/models/blocks.py:236-239)
    if (f3r_layernorm(x, b.norm1_w, b.norm1_b, h, 0, rows, dim, eps, stream)) return 1;
    f3r_gemm_desc d;
    memset(&d, 0, sizeof(d));
    d.a = h; d.wt = b.qkv_w; d.n = 3 * dim; d.k = dim; d.taps = 1; d.w = rows; d.h = 1; d.nb = 1; d.a_ld = dim;
    d.bias = b.qkv_b; d.out0 = q; d.ldo = dim; d.split_col = dim; d.out0b = kv; d.ldo_b = 2 * dim;
    if (rope) {
      d.epi = F3R_EPI_ROPE; d.tok_per_img = rope_tok_per_img; d.grid_w = rope_grid_w; d.rope_cols = 2 * dim;
      d.rope_cos = rope_cos; d.rope_sin = rope_sin;
    }
    if (f3r_gemm(&d, stream)) return 1;
    if (f3r_attention(q, dim, kv, 2 * dim, att, dim, nullptr, batch, heads, seq, seq, scale, stream)) return 1;
    memset(&d, 0, sizeof(d));
    d.a = att; d.wt = b.proj_w; d.n = dim; d.k = dim; d.taps = 1; d.w = rows; d.h = 1; d.nb = 1; d.a_ld = dim;
    d.bias = b.proj_b; d.out0 = x; d.out0_f32 = 1; d.res0 = x; d.res0_f32 = 1; d.ldo = dim;
    if (f3r_gemm(&d, stream)) return 1;
    if (f3r_layernorm(x, b.norm2_w, b.norm2_b, h, 0, rows, dim, eps, stream)) return 1;
    memset(&d, 0, sizeof(d));
    d.a = h; d.wt = b.fc1_w; d.n = hidden; d.k = dim; d.taps = 1; d.w = rows; d.h = 1; d.nb = 1; d.a_ld = dim;
    d.bias = b.fc1_b; d.out0 = hid; d.ldo = hidden; d.act = F3R_ACT_GELU;
    if (f3r_gemm(&d, stream)) return 1;
    memset(&d, 0, sizeof(d));
    d.a = hid; d.wt = b.fc2_w; d.n = dim; d.k = hidden; d.taps = 1; d.w = rows; d.h = 1; d.nb = 1; d.a_ld = hidden;
    d.bias = b.fc2_b; d.out0 = x; d.out0_f32 = 1; d.res0 = x; d.res0_f32 = 1; d.ldo = dim;
    if (f3r_gemm(&d, stream)) return 1;
  }
  return 0;
}

int f3r_cast_bf16(const float* in, void* out, size_t count, void* stream) {
  if (!in || !out) return fail("f3r_cast_bf16: null operand");
  g_launches++;
  return check(f3r::launch_cast_bf16(in, out, count, static_cast<cudaStream_t>(stream)), "f3r_cast_bf16");
}

}  // extern "C"
