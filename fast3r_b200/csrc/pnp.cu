// Camera pose of every view from its pointmap: batched P3P-RANSAC with an optional focal sweep, then a Levenberg-Marquardt
// refit on the inliers - what fast_pnp (fast3r/dust3r/cloud_opt/init_im_poses.py:300-350) does per view and per focal
// with cv2.solvePnPRansac.  One stream-ordered pipeline over all views of one shape:
//   compact    indices of the masked pixels of each view, in pixel order, and their count m
//   hypotheses one per (view, focal k, iteration i): 4 distinct list entries from a counter-based hash (pnp_math.h),
//              P3P on the first three, the solution that reprojects the fourth best; P = K [R | t] stored as 12 floats
//   score      inlier count of every hypothesis over every masked pixel (the hot kernel, FMA-pipe bound)
//   select     per view the highest score, ties to the lowest (k, i)
//   refit      PNP_LM_STEPS Levenberg-Marquardt steps on the reprojection error over the selected hypothesis's inliers
// Counts are integers and every fp64 reduction runs in a fixed order, so the result does not depend on scheduling, on
// the other views of the call or on the position of a view in it.
#include <math.h>

#include "f3r_kernels.h"
#include "pnp_math.h"

namespace f3r {

namespace {

constexpr int CMP_THREADS = 1024;
constexpr int HYP_THREADS = 128;
constexpr int SC_THREADS = 256;
constexpr int SC_PPT = 8;                         // masked pixels per thread, held in registers
constexpr int SC_TILE = SC_THREADS * SC_PPT;      // masked pixels per CTA
constexpr int SC_CHUNK = 128;                     // hypotheses staged in shared memory at a time
constexpr int LM_THREADS = 256;
constexpr int LM_CHUNKS = 32;                     // partial sums per view (fixed, so the reduction order is)
constexpr int LM_VALS = 29;                       // J^T J upper triangle (21), J^T r (6), cost, points behind the camera
constexpr int LM_STEPS = PNP_LM_STEPS;
constexpr int ST_CUR = 0, ST_TRIAL = 12, ST_COST = 24, ST_JTJ = 25, ST_JTR = 46, ST_LAMBDA = 52, ST_SIZE = 56;

__device__ __forceinline__ float4 ld_pt(const float* __restrict__ pts, size_t view_base, int pix) {
  const float* p = pts + (view_base + static_cast<size_t>(pix)) * 3;
  return make_float4(p[0], p[1], p[2], 0.f);
}

// (P0 X - u P2 X)^2 + (P1 X - v P2 X)^2 <= 25 (P2 X)^2 in fp32, division-free.  P2 X == 0 and NaN are not inliers;
// otherwise the same as a reprojection error <= 5 px.  Written with explicit roundings so every kernel evaluates the same
// set.
__device__ __forceinline__ bool inlier(const float* P, float x, float y, float z, float u, float v) {
  const float w = fmaf(P[8], x, fmaf(P[9], y, fmaf(P[10], z, P[11])));
  const float a = fmaf(P[0], x, fmaf(P[1], y, fmaf(P[2], z, P[3])));
  const float b = fmaf(P[4], x, fmaf(P[5], y, fmaf(P[6], z, P[7])));
  const float e0 = fmaf(-u, w, a), e1 = fmaf(-v, w, b);
  const float lhs = fmaf(e1, e1, __fmul_rn(e0, e0));
  return lhs <= __fmul_rn(25.f, __fmul_rn(w, w)) && w != 0.f;
}

// One CTA per view: stream compaction of the mask in pixel order (ballot + warp prefix + block scan per 1024 pixels).
__global__ void __launch_bounds__(CMP_THREADS) pnp_compact_kernel(const uint8_t* __restrict__ mask, int n,
                                                                  int* __restrict__ idx, int* __restrict__ count) {
  __shared__ int warp_tot[CMP_THREADS / 32];
  __shared__ int s_base;
  const int view = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const uint8_t* mv = mask + static_cast<size_t>(view) * n;
  int* iv = idx + static_cast<size_t>(view) * n;
  if (tid == 0) s_base = 0;
  __syncthreads();
  for (int base = 0; base < n; base += CMP_THREADS) {
    const int i = base + tid;
    const bool f = i < n && mv[i] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) warp_tot[wid] = __popc(bal);
    __syncthreads();
    if (wid == 0) {
      const int t = warp_tot[lane];
      int s = t;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, s, o);
        if (lane >= o) s += y;
      }
      warp_tot[lane] = s - t;  // exclusive
    }
    __syncthreads();
    const int b0 = s_base;
    if (f) iv[b0 + warp_tot[wid] + __popc(bal & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (tid == CMP_THREADS - 1) s_base = b0 + warp_tot[wid] + __popc(bal);
    __syncthreads();
  }
  if (tid == 0) count[view] = s_base;
}

__device__ __forceinline__ void view_camera(const float* focals, int n_focals, const float* pp, int view, int k, int H,
                                            int W, double& f, double& cx, double& cy) {
  f = focals[static_cast<size_t>(view) * n_focals + k];
  cx = pp ? pp[2 * view] : 0.5f * static_cast<float>(W);
  cy = pp ? pp[2 * view + 1] : 0.5f * static_cast<float>(H);
}

// One thread per (view, k, i).  An invalid hypothesis gets a NaN P (it counts no inlier).
__global__ void __launch_bounds__(HYP_THREADS) pnp_hypothesis_kernel(
    const float* __restrict__ pts, const int* __restrict__ idx, const int* __restrict__ count, int views, int H, int W,
    const float* __restrict__ focals, int n_focals, const float* __restrict__ pp, int iters, float* __restrict__ hypP,
    double* __restrict__ hyp_pose) {
  const int hyps = n_focals * iters;
  const long g = static_cast<long>(blockIdx.x) * HYP_THREADS + threadIdx.x;
  if (g >= static_cast<long>(views) * hyps) return;
  const int view = static_cast<int>(g / hyps), h = static_cast<int>(g % hyps), k = h / iters, it = h % iters;
  const int n = H * W;
  double f, cx, cy;
  view_camera(focals, n_focals, pp, view, k, H, W, f, cx, cy);
  uint32_t e[4];
  double pose[12], P[12];
  bool ok = pnp_sample4(static_cast<uint32_t>(count[view]), static_cast<uint32_t>(k), static_cast<uint32_t>(it), e);
  if (ok) {
    double X[4][3], uv[4][2];
    const size_t vb = static_cast<size_t>(view) * n;
    for (int j = 0; j < 4; ++j) {
      const int pix = idx[vb + e[j]];
      const float4 p = ld_pt(pts, vb, pix);
      X[j][0] = p.x; X[j][1] = p.y; X[j][2] = p.z;
      uv[j][0] = pix % W; uv[j][1] = pix / W;
      ok &= isfinite(p.x) && isfinite(p.y) && isfinite(p.z);
    }
    ok = ok && p3p_hypothesis(X, uv, f, cx, cy, pose);
  }
  if (ok) projection_matrix(pose, f, cx, cy, P);
  float* out = hypP + static_cast<size_t>(g) * 12;
  double* outp = hyp_pose + static_cast<size_t>(g) * 12;
  for (int j = 0; j < 12; ++j) {
    out[j] = ok ? static_cast<float>(P[j]) : __int_as_float(0x7fffffff);
    outp[j] = ok ? pose[j] : 0.0;
  }
}

// grid (tiles of SC_TILE masked pixels, view).  Each thread keeps SC_PPT pixels in registers; the view's hypotheses
// stream through shared memory; per hypothesis a warp sum, a shared atomic per warp and one global atomic per CTA.
__global__ void __launch_bounds__(SC_THREADS) pnp_score_kernel(const float* __restrict__ pts, const int* __restrict__ idx,
                                                               const int* __restrict__ count, int W, int n,
                                                               const float* __restrict__ hypP, int hyps,
                                                               int32_t* __restrict__ scores) {
  __shared__ __align__(16) float sP[SC_CHUNK][12];
  __shared__ int sCnt[SC_CHUNK];
  const int view = blockIdx.y, tid = threadIdx.x;
  const int m = count[view];
  const int t0 = blockIdx.x * SC_TILE;
  if (t0 >= m) return;
  const size_t vb = static_cast<size_t>(view) * n;
  float px[SC_PPT], py[SC_PPT], pz[SC_PPT], pu[SC_PPT], pv[SC_PPT];
#pragma unroll
  for (int j = 0; j < SC_PPT; ++j) {
    const int e = t0 + j * SC_THREADS + tid;
    if (e < m) {
      const int pix = idx[vb + e];
      const float4 p = ld_pt(pts, vb, pix);
      px[j] = p.x; py[j] = p.y; pz[j] = p.z;
      pu[j] = static_cast<float>(pix % W);
      pv[j] = static_cast<float>(pix / W);
    } else {
      px[j] = py[j] = pz[j] = __int_as_float(0x7fffffff);  // NaN: never an inlier
      pu[j] = pv[j] = 0.f;
    }
  }
  const float* hv = hypP + static_cast<size_t>(view) * hyps * 12;
  int32_t* sv = scores + static_cast<size_t>(view) * hyps;
  for (int c0 = 0; c0 < hyps; c0 += SC_CHUNK) {
    const int nc = min(SC_CHUNK, hyps - c0);
    for (int j = tid; j < nc * 12; j += SC_THREADS) sP[j / 12][j % 12] = hv[static_cast<size_t>(c0) * 12 + j];
    for (int j = tid; j < SC_CHUNK; j += SC_THREADS) sCnt[j] = 0;
    __syncthreads();
    for (int h = 0; h < nc; ++h) {
      float P[12];
      const float4* s4 = reinterpret_cast<const float4*>(sP[h]);
      const float4 q0 = s4[0], q1 = s4[1], q2 = s4[2];
      P[0] = q0.x; P[1] = q0.y; P[2] = q0.z; P[3] = q0.w; P[4] = q1.x; P[5] = q1.y;
      P[6] = q1.z; P[7] = q1.w; P[8] = q2.x; P[9] = q2.y; P[10] = q2.z; P[11] = q2.w;
      int c = 0;
#pragma unroll
      for (int j = 0; j < SC_PPT; ++j) c += inlier(P, px[j], py[j], pz[j], pu[j], pv[j]) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if ((tid & 31) == 0 && c) atomicAdd(&sCnt[h], c);
    }
    __syncthreads();
    for (int j = tid; j < nc; j += SC_THREADS)
      if (sCnt[j]) atomicAdd(&sv[c0 + j], sCnt[j]);
    __syncthreads();
  }
}

// One CTA per view: best = argmax score (ties to the lowest flat index k * iters + i); the refit starts from its pose.
__global__ void __launch_bounds__(256) pnp_select_kernel(const int32_t* __restrict__ scores, int hyps, int iters,
                                                         const double* __restrict__ hyp_pose, int32_t* __restrict__ best,
                                                         double* __restrict__ state, double* __restrict__ c2w) {
  __shared__ long long red[8];
  const int view = blockIdx.x, tid = threadIdx.x;
  long long key = -1;  // (score << 32) | (2^31 - 1 - h): the maximum is the highest score, then the lowest h
  for (int h = tid; h < hyps; h += 256) {
    const long long s = scores[static_cast<size_t>(view) * hyps + h];
    const long long kk = (s << 32) | static_cast<long long>(0x7fffffff - h);
    key = kk > key ? kk : key;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const long long y = __shfl_down_sync(0xffffffffu, key, o);
    key = y > key ? y : key;
  }
  if ((tid & 31) == 0) red[tid >> 5] = key;
  __syncthreads();
  if (tid != 0) return;
  for (int w = 1; w < 8; ++w) key = red[w] > key ? red[w] : key;
  double* st = state + static_cast<size_t>(view) * ST_SIZE;
  if ((key >> 32) <= 0) {
    best[2 * view] = best[2 * view + 1] = -1;
    for (int j = 0; j < 12; ++j) c2w[static_cast<size_t>(view) * 12 + j] = 0.0;
    return;
  }
  const int h = 0x7fffffff - static_cast<int>(key & 0xffffffffll);
  best[2 * view] = h / iters;
  best[2 * view + 1] = h % iters;
  for (int j = 0; j < 12; ++j) st[ST_TRIAL + j] = hyp_pose[(static_cast<size_t>(view) * hyps + h) * 12 + j];
}

// One refit pass at the trial pose, over the inliers of the selected hypothesis: fp64 J^T J, J^T r and cost per chunk.
__global__ void __launch_bounds__(LM_THREADS) pnp_lm_pass_kernel(
    const float* __restrict__ pts, const int* __restrict__ idx, const int* __restrict__ count, int H, int W,
    const float* __restrict__ focals, int n_focals, const float* __restrict__ pp, int iters,
    const float* __restrict__ hypP, const int32_t* __restrict__ best, const double* __restrict__ state,
    double* __restrict__ partial) {
  __shared__ double red[LM_THREADS / 32][LM_VALS];
  const int view = blockIdx.y, chunk = blockIdx.x, tid = threadIdx.x;
  const int k = best[2 * view];
  if (k < 0) return;
  const int hyps = n_focals * iters;
  const int h = k * iters + best[2 * view + 1];
  const int n = H * W, m = count[view];
  const size_t vb = static_cast<size_t>(view) * n;
  float P[12];
  for (int j = 0; j < 12; ++j) P[j] = hypP[(static_cast<size_t>(view) * hyps + h) * 12 + j];
  double f, cx, cy;
  view_camera(focals, n_focals, pp, view, k, H, W, f, cx, cy);
  const double* T = state + static_cast<size_t>(view) * ST_SIZE + ST_TRIAL;
  double R[9], t[3];
  for (int j = 0; j < 9; ++j) R[j] = T[j];
  for (int j = 0; j < 3; ++j) t[j] = T[9 + j];
  double acc[LM_VALS];
#pragma unroll
  for (int j = 0; j < LM_VALS; ++j) acc[j] = 0.0;
  const int per = (m + LM_CHUNKS - 1) / LM_CHUNKS;
  const int e0 = min(m, chunk * per), e1 = min(m, e0 + per);
  for (int e = e0 + tid; e < e1; e += LM_THREADS) {
    const int pix = idx[vb + e];
    const float4 p = ld_pt(pts, vb, pix);
    const float u = static_cast<float>(pix % W), v = static_cast<float>(pix / W);
    if (!inlier(P, p.x, p.y, p.z, u, v)) continue;
    const double X[3] = {p.x, p.y, p.z};
    const double q[3] = {R[0] * X[0] + R[1] * X[1] + R[2] * X[2], R[3] * X[0] + R[4] * X[1] + R[5] * X[2],
                         R[6] * X[0] + R[7] * X[1] + R[8] * X[2]};
    const double xc = q[0] + t[0], yc = q[1] + t[1], zc = q[2] + t[2];
    if (!(zc > 0.0)) {
      acc[28] += 1.0;
      continue;
    }
    const double iz = 1.0 / zc;
    const double ru = f * xc * iz + cx - u, rv = f * yc * iz + cy - v;
    // d(u, v)/dXc and dXc/d(w, dt) = (-[q]x, I)
    const double gx = f * iz, gzu = -f * xc * iz * iz, gzv = -f * yc * iz * iz;
    const double Ju[6] = {gzu * q[1], gx * q[2] - gzu * q[0], -gx * q[1], gx, 0.0, gzu};
    const double Jv[6] = {-gx * q[2] + gzv * q[1], -gzv * q[0], gx * q[0], 0.0, gx, gzv};
    int c = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
      for (int b = a; b < 6; ++b) acc[c++] += Ju[a] * Ju[b] + Jv[a] * Jv[b];
    }
#pragma unroll
    for (int a = 0; a < 6; ++a) acc[21 + a] += Ju[a] * ru + Jv[a] * rv;
    acc[27] += ru * ru + rv * rv;
  }
#pragma unroll
  for (int j = 0; j < LM_VALS; ++j) {
    double va = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) va += __shfl_down_sync(0xffffffffu, va, o);
    if ((tid & 31) == 0) red[tid >> 5][j] = va;
  }
  __syncthreads();
  if (tid < LM_VALS) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < LM_THREADS / 32; ++w) s += red[w][tid];
    partial[(static_cast<size_t>(view) * LM_CHUNKS + chunk) * LM_VALS + tid] = s;
  }
}

// One thread per view: accept the trial pose if it lowers the cost (step 0: always, it is the P3P pose), adapt the
// damping, and either propose the next trial (Marquardt-damped normal equations) or, after the last pass, write c2w.
__global__ void pnp_lm_solve_kernel(const double* __restrict__ partial, const int32_t* __restrict__ best, int views,
                                    int step, int last, double* __restrict__ state, double* __restrict__ c2w) {
  const int view = blockIdx.x * blockDim.x + threadIdx.x;
  if (view >= views || best[2 * view] < 0) return;
  double tot[LM_VALS];
  for (int j = 0; j < LM_VALS; ++j) tot[j] = 0.0;
  for (int c = 0; c < LM_CHUNKS; ++c)
    for (int j = 0; j < LM_VALS; ++j) tot[j] += partial[(static_cast<size_t>(view) * LM_CHUNKS + c) * LM_VALS + j];
  double* st = state + static_cast<size_t>(view) * ST_SIZE;
  const double cost = (tot[28] == 0.0 && isfinite(tot[27])) ? tot[27] : INFINITY;
  const bool accept = step == 0 || cost < st[ST_COST];
  if (accept) {
    for (int j = 0; j < 12; ++j) st[ST_CUR + j] = st[ST_TRIAL + j];
    st[ST_COST] = cost;
    for (int j = 0; j < 27; ++j) st[ST_JTJ + j] = tot[j];
    st[ST_LAMBDA] = step == 0 ? 1e-3 : fmax(st[ST_LAMBDA] * 0.1, 1e-12);
  } else {
    st[ST_LAMBDA] = fmin(st[ST_LAMBDA] * 10.0, 1e12);
  }
  if (last) {
    pose_inverse(st + ST_CUR, c2w + static_cast<size_t>(view) * 12);
    return;
  }
  double A[21], rhs[6], d[6];
  const int diag[6] = {0, 6, 11, 15, 18, 20};
  for (int j = 0; j < 21; ++j) A[j] = st[ST_JTJ + j];
  for (int a = 0; a < 6; ++a) {
    A[diag[a]] *= 1.0 + st[ST_LAMBDA];
    rhs[a] = -st[ST_JTR + a];
  }
  if (chol6_solve(A, rhs, d)) {
    pose_update(st + ST_CUR, d, st + ST_TRIAL);
  } else {
    for (int j = 0; j < 12; ++j) st[ST_TRIAL + j] = st[ST_CUR + j];
  }
}

size_t al256(size_t b) { return (b + 255) & ~static_cast<size_t>(255); }

}  // namespace

// idx int32 [views][n] | count int32 [views] | hypothesis P fp32 [views][hyps][12] | hypothesis pose fp64 [views][hyps][12]
// | refit partial sums fp64 [views][LM_CHUNKS][LM_VALS] | refit state fp64 [views][ST_SIZE], each part 256-byte aligned
size_t pnp_workspace(int views, int n, int hyps) {
  const size_t v = static_cast<size_t>(views);
  return al256(v * n * 4) + al256(v * 4) + al256(v * hyps * 12 * 4) + al256(v * hyps * 12 * 8) +
         al256(v * LM_CHUNKS * LM_VALS * 8) + al256(v * ST_SIZE * 8);
}

cudaError_t launch_pnp_ransac(const float* pts, const uint8_t* mask, int views, int H, int W, const float* focals,
                              int n_focals, const float* pp, int iters, int32_t* scores, int32_t* best, double* c2w,
                              void* workspace, cudaStream_t stream) {
  const int n = H * W, hyps = n_focals * iters;
  const size_t v = static_cast<size_t>(views);
  uint8_t* w = static_cast<uint8_t*>(workspace);
  int* idx = reinterpret_cast<int*>(w);
  w += al256(v * n * 4);
  int* count = reinterpret_cast<int*>(w);
  w += al256(v * 4);
  float* hypP = reinterpret_cast<float*>(w);
  w += al256(v * hyps * 12 * 4);
  double* hyp_pose = reinterpret_cast<double*>(w);
  w += al256(v * hyps * 12 * 8);
  double* partial = reinterpret_cast<double*>(w);
  w += al256(v * LM_CHUNKS * LM_VALS * 8);
  double* state = reinterpret_cast<double*>(w);

  cudaError_t e = cudaMemsetAsync(scores, 0, v * hyps * sizeof(int32_t), stream);
  if (e != cudaSuccess) return e;
  pnp_compact_kernel<<<views, CMP_THREADS, 0, stream>>>(mask, n, idx, count);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const long nh = static_cast<long>(views) * hyps;
  pnp_hypothesis_kernel<<<static_cast<unsigned>((nh + HYP_THREADS - 1) / HYP_THREADS), HYP_THREADS, 0, stream>>>(
      pts, idx, count, views, H, W, focals, n_focals, pp, iters, hypP, hyp_pose);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  pnp_score_kernel<<<dim3((n + SC_TILE - 1) / SC_TILE, views), SC_THREADS, 0, stream>>>(pts, idx, count, W, n, hypP, hyps,
                                                                                         scores);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  pnp_select_kernel<<<views, 256, 0, stream>>>(scores, hyps, iters, hyp_pose, best, state, c2w);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  for (int s = 0; s <= LM_STEPS; ++s) {
    pnp_lm_pass_kernel<<<dim3(LM_CHUNKS, views), LM_THREADS, 0, stream>>>(pts, idx, count, H, W, focals, n_focals, pp,
                                                                          iters, hypP, best, state, partial);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    pnp_lm_solve_kernel<<<(views + 31) / 32, 32, 0, stream>>>(partial, best, views, s, s == LM_STEPS, state, c2w);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return cudaSuccess;
}

}  // namespace f3r
