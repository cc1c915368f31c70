// loss.cu -- tiled pairwise-L2 arg-min and the probabilistic chamfer reduction.
// Reference: models/losses.py:50-99 (ChamferLoss_Brute), :125-143 (SingleSideChamferLoss_Brute),
// models/keypoint_detector.py:182-197.
#include "common.cuh"
#include "desc_dist.cuh"

namespace usip {

constexpr int PM_THREADS = 256;
constexpr int PM_Q = 128;       // queries per CTA (two threads per query, each on half of the tile)
constexpr int PM_TILE = 512;    // database points staged per CTA (float4 each -> 8 KB)

__global__ void pm_init_kernel(unsigned long long* packed, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) packed[i] = ~0ull;
}

// grid (ceil(Nb/PM_TILE), ceil(Ma/PM_Q), B): thread = (query, tile half); partial results merge through a 64-bit
// atomicMin on (d2 bits << 32 | j), which yields the first index among exact ties (d2 >= 0 so float bits order like
// uints).  Small tiles keep the per-thread dependent min chain short and put >1000 CTAs on the machine.
__global__ void __launch_bounds__(PM_THREADS)
pairwise_min_kernel(const float* __restrict__ a, const float* __restrict__ b,
                    unsigned long long* __restrict__ packed, int Ma, int Nb) {
  __shared__ float4 sb[PM_TILE];
  const int bb = blockIdx.z;
  const int i = blockIdx.y * PM_Q + (threadIdx.x & (PM_Q - 1));
  const int hf = threadIdx.x >> 7;
  const int j0 = blockIdx.x * PM_TILE;
  const int jc = min(PM_TILE, Nb - j0);
  const float* pb = b + (size_t)bb * 3 * Nb;
  for (int t = threadIdx.x; t < jc; t += PM_THREADS)
    sb[t] = make_float4(pb[j0 + t], pb[Nb + j0 + t], pb[2 * Nb + j0 + t], 0.f);
  __syncthreads();
  if (i >= Ma) return;
  const float* pa = a + (size_t)bb * 3 * Ma;
  const float ax = pa[i], ay = pa[Ma + i], az = pa[2 * Ma + i];
  const int t0 = hf * (PM_TILE / 2), t1 = min(jc, t0 + PM_TILE / 2);
  float best0 = INFINITY, best1 = INFINITY; int bj0 = 0, bj1 = 0;
  int t = t0;
  for (; t + 1 < t1; t += 2) {                       // two independent chains
    const float4 q0 = sb[t], q1 = sb[t + 1];
    const float d0 = sqdist_rn(ax, ay, az, q0.x, q0.y, q0.z), d1 = sqdist_rn(ax, ay, az, q1.x, q1.y, q1.z);
    if (d0 < best0) { best0 = d0; bj0 = t; }
    if (d1 < best1) { best1 = d1; bj1 = t + 1; }
  }
  if (t < t1) { const float4 q0 = sb[t]; const float d0 = sqdist_rn(ax, ay, az, q0.x, q0.y, q0.z); if (d0 < best0) { best0 = d0; bj0 = t; } }
  // merge the chains: smaller distance, then smaller index
  float best = best0; int bj = bj0;
  if (best1 < best || (best1 == best && bj1 < bj)) { best = best1; bj = bj1; }
  if (best == best && best < INFINITY) {
    unsigned long long key = ((unsigned long long)__float_as_uint(best) << 32) | (unsigned)(j0 + bj);
    atomicMin(&packed[(size_t)bb * Ma + i], key);
  }
}

// Direct variant: one CTA owns Q queries (256 / Q threads per query, each on its slice of every tile) and walks ALL
// database tiles, so there is no cross-CTA merge and no init / finish launch.  Used for small databases (the keypoint
// <-> keypoint chamfer searches, Q = 128).  For keypoints against a whole cloud the split-database kernel above stays:
// a direct Q = 32 variant (128 CTAs of 8 warps walking 32 tiles each) measured 82 us against 61 us -- too few warps
// per SM to hide the shared-memory latency.  Same arithmetic and tie rule: smaller distance, then smaller index.
template <int Q>
__global__ void __launch_bounds__(PM_THREADS)
pairwise_min_direct_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ min_d,
                           int32_t* __restrict__ arg, int Ma, int Nb) {
  constexpr int SL = PM_THREADS / Q;               // slices per query
  constexpr int SPAN = PM_TILE / SL;               // database points per slice and tile
  __shared__ float4 sb[PM_TILE];
  __shared__ float hbest[SL][Q]; __shared__ int hidx[SL][Q];
  const int bb = blockIdx.y;
  const int q = threadIdx.x % Q, sl = threadIdx.x / Q;
  const int i = blockIdx.x * Q + q;
  const float* pa = a + (size_t)bb * 3 * Ma; const float* pb = b + (size_t)bb * 3 * Nb;
  const bool ok = i < Ma;
  const float ax = ok ? pa[i] : 0.f, ay = ok ? pa[Ma + i] : 0.f, az = ok ? pa[2 * Ma + i] : 0.f;
  float best0 = INFINITY, best1 = INFINITY; int bj0 = 0, bj1 = 0;
  for (int j0 = 0; j0 < Nb; j0 += PM_TILE) {
    const int jc = min(PM_TILE, Nb - j0);
    __syncthreads();
    for (int t = threadIdx.x; t < jc; t += PM_THREADS) sb[t] = make_float4(pb[j0 + t], pb[Nb + j0 + t], pb[2 * Nb + j0 + t], 0.f);
    __syncthreads();
    const int t0 = sl * SPAN, t1 = min(jc, t0 + SPAN);
    int t = t0;
    for (; t + 1 < t1; t += 2) {                   // two independent chains; ascending j inside each: '<' keeps the first minimum
      const float4 p0 = sb[t], p1 = sb[t + 1];
      const float d0 = sqdist_rn(ax, ay, az, p0.x, p0.y, p0.z), d1 = sqdist_rn(ax, ay, az, p1.x, p1.y, p1.z);
      if (d0 < best0) { best0 = d0; bj0 = j0 + t; }
      if (d1 < best1) { best1 = d1; bj1 = j0 + t + 1; }
    }
    if (t < t1) { const float4 p0 = sb[t]; const float d0 = sqdist_rn(ax, ay, az, p0.x, p0.y, p0.z); if (d0 < best0) { best0 = d0; bj0 = j0 + t; } }
  }
  float best = best0; int bj = bj0;
  if (best1 < best || (best1 == best && bj1 < bj)) { best = best1; bj = bj1; }
  hbest[sl][q] = best; hidx[sl][q] = bj;
  __syncthreads();
  if (sl == 0 && ok) {
#pragma unroll
    for (int s2 = 1; s2 < SL; ++s2) {
      const float ob = hbest[s2][q]; const int oj = hidx[s2][q];
      if (ob < best || (ob == best && oj < bj)) { best = ob; bj = oj; }
    }
    const bool none = !(best < INFINITY);
    const size_t o = (size_t)bb * Ma + i;
    if (min_d) min_d[o] = none ? INFINITY : __fsqrt_rn(best);
    if (arg) arg[o] = none ? 0 : bj;
  }
}

__global__ void pm_finish_kernel(const unsigned long long* __restrict__ packed, float* __restrict__ min_d,
                                 int32_t* __restrict__ arg, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long k = packed[i];
  bool none = (k == ~0ull);
  float d2 = __uint_as_float((unsigned)(k >> 32));
  if (min_d) min_d[i] = none ? INFINITY : __fsqrt_rn(d2);     // torch.norm = sqrt of the fp32 sum
  if (arg) arg[i] = none ? 0 : (int32_t)(k & 0xffffffffull);
}

// block-wide deterministic double sum
__device__ double block_sum(double v, double* sh) {
  v = warp_sum_d(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x == 0) for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += sh[i];
  return r;   // valid on thread 0
}

// losses.py:79-97.  Single CTA (sizes are B*M ~ 1e4).  Per-element arithmetic in fp32 like the reference (log, divide),
// sums in fp64; the eight sums are reduced together (one barrier).
__global__ void __launch_bounds__(1024)
chamfer_prob_reduce_kernel(const float* __restrict__ d_sd, const int32_t* __restrict__ i_sd,
                           const float* __restrict__ d_ds, const int32_t* __restrict__ i_ds,
                           const float* __restrict__ sig_src, const float* __restrict__ sig_dst,
                           float* __restrict__ out3, int B, int M, int N) {
  __shared__ double sh[8][32];
  double r[8] = {0, 0, 0, 0, 0, 0, 0, 0};          // forward: loss, d, 1/s, d/s; backward: the same
  // four elements per thread and pass: the index -> sigma gathers are two dependent loads per element, so the loads of a
  // batch are issued together (B*M = 4096 elements on 1024 threads: one batch per direction instead of four round trips)
  auto side = [&](const float* dd, const int32_t* ii, const float* s_own, const float* s_other, int n_own, int n_other, int q0) {
    const int total = B * n_own;
    for (int t0 = threadIdx.x; t0 < total; t0 += 4 * blockDim.x) {
      int idx[4]; float so[4], d[4], sg[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = t0 + u * blockDim.x; const bool ok = t < total;
        idx[u] = ok ? ii[t] : 0; so[u] = ok ? s_own[t] : 1.f; d[u] = ok ? dd[t] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int t = t0 + u * blockDim.x;
        sg[u] = t < total ? s_other[(size_t)(t / n_own) * n_other + idx[u]] : 1.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (t0 + u * (int)blockDim.x < total) {
          const float s = 0.5f * (so[u] + sg[u]);
          const float ds = d[u] / s;
          r[q0 + 0] += (double)(logf(s) + ds); r[q0 + 1] += (double)d[u]; r[q0 + 2] += (double)(1.0f / s); r[q0 + 3] += (double)ds;
        }
      }
    }
  };
  side(d_sd, i_sd, sig_src, sig_dst, M, N, 0);
  side(d_ds, i_ds, sig_dst, sig_src, N, M, 4);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int q = 0; q < 8; ++q) { r[q] = warp_sum_d(r[q]); if (lane == 0) sh[q][w] = r[q]; }
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int q = 0; q < 8; ++q) r[q] = warp_sum_d(lane < (int)(blockDim.x >> 5) ? sh[q][lane] : 0.0);
    if (lane == 0) {
      const double nf = (double)B * M, nb = (double)B * N;
      out3[0] = (float)(r[0] / nf + r[4] / nb);
      out3[1] = (float)(r[1] / nf + r[5] / nb);
      // mean(w*d), w = (1/s)/mean(1/s)  ==  mean(d/s) / mean(1/s)
      out3[2] = (float)((r[3] / nf) / (r[2] / nf) + (r[7] / nb) / (r[6] / nb));
    }
  }
}

__global__ void transform_points_kernel(const float* __restrict__ kp, const float* __restrict__ R,
                                        const float* __restrict__ scale, const float* __restrict__ shift,
                                        float* __restrict__ out, int B, int M) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * M) return;
  int b = t / M, m = t - b * M;
  const float* p = kp + (size_t)b * 3 * M;
  const float x = p[m], y = p[M + m], z = p[2 * M + m];
  const float* r = R + (size_t)b * 9;
  const float s = scale[b];
  for (int c = 0; c < 3; ++c) {
    float v = r[c * 3 + 0] * x + r[c * 3 + 1] * y + r[c * 3 + 2] * z;   // torch.matmul(R, kp)
    out[(size_t)b * 3 * M + (size_t)c * M + m] = v * s + shift[b * 3 + c];
  }
}

__global__ void __launch_bounds__(1024)
mean_scale_kernel(const float* __restrict__ d, int64_t n, float alpha, float* __restrict__ out) {
  __shared__ double sh[32];
  double s = 0;
  for (int64_t t = threadIdx.x; t < n; t += blockDim.x) s += d[t];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) out[0] = (float)(s / (double)n) * alpha;
}


// ---- backward kernels -------------------------------------------------------------------------
// d/da_i ||a_i - b_j*|| = (a_i - b_j*)/d  (0 at d == 0, torch.norm's sub-gradient; losses.py:65)
__global__ void pairwise_min_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                        const float* __restrict__ min_d, const int32_t* __restrict__ arg,
                                        const float* __restrict__ g, float gscale, float* __restrict__ ga,
                                        float* __restrict__ gb, int B, int Ma, int Nb) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * Ma) return;
  int bb = t / Ma, i = t - bb * Ma;
  int j = arg[t];
  float d = min_d[t];
  float gi = (g ? g[t] : 1.f) * gscale;
  float inv = d > 0.f ? gi / d : 0.f;
  const float* pa = a + (size_t)bb * 3 * Ma; const float* pb = b + (size_t)bb * 3 * Nb;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float diff = pa[(size_t)c * Ma + i] - pb[(size_t)c * Nb + j];
    float v = diff * inv;
    if (ga) ga[(size_t)bb * 3 * Ma + (size_t)c * Ma + i] = v;
    if (gb) atomicAdd(&gb[(size_t)bb * 3 * Nb + (size_t)c * Nb + j], -v);
  }
}

// backward of ChamferLoss_Brute's sigma branch (losses.py:79-90); all grads accumulate atomically into
// pre-zeroed buffers.  dir 0: src->dst terms, dir 1: dst->src terms.
__global__ void chamfer_prob_bwd_kernel(const float* __restrict__ src, const float* __restrict__ dst,
                                        const float* __restrict__ sig_src, const float* __restrict__ sig_dst,
                                        const float* __restrict__ d_sd, const int32_t* __restrict__ i_sd,
                                        const float* __restrict__ d_ds, const int32_t* __restrict__ i_ds,
                                        const float* __restrict__ gout, float* __restrict__ g_src,
                                        float* __restrict__ g_dst, float* __restrict__ g_ss, float* __restrict__ g_sd,
                                        int B, int M, int N) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int nf = B * M, nb = B * N;
  if (t >= nf + nb) return;
  const float go = gout[0];
  const bool fwd = t < nf;
  const int u = fwd ? t : t - nf;
  const int La = fwd ? M : N, Lb = fwd ? N : M;            // a = own set, b = other set
  const int bb = u / La, i = u - bb * La;
  const float* A = fwd ? src : dst; const float* Bm = fwd ? dst : src;
  const float* sa = fwd ? sig_src : sig_dst; const float* sb = fwd ? sig_dst : sig_src;
  float* gA = fwd ? g_src : g_dst; float* gB = fwd ? g_dst : g_src;
  float* gsa = fwd ? g_ss : g_sd; float* gsb = fwd ? g_sd : g_ss;
  const int j = fwd ? i_sd[u] : i_ds[u];
  const float d = fwd ? d_sd[u] : d_ds[u];
  const float s = 0.5f * (sa[(size_t)bb * La + i] + sb[(size_t)bb * Lb + j]);
  const float w = go / (float)(fwd ? nf : nb);
  const float gd = w / s;                                   // d loss / d d
  const float gs = w * (1.f / s - d / (s * s)) * 0.5f;      // d loss / d sigma (each of the two)
  atomicAdd(&gsa[(size_t)bb * La + i], gs);
  atomicAdd(&gsb[(size_t)bb * Lb + j], gs);
  const float inv = d > 0.f ? gd / d : 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float diff = A[(size_t)bb * 3 * La + (size_t)c * La + i] - Bm[(size_t)bb * 3 * Lb + (size_t)c * Lb + j];
    atomicAdd(&gA[(size_t)bb * 3 * La + (size_t)c * La + i], diff * inv);
    atomicAdd(&gB[(size_t)bb * 3 * Lb + (size_t)c * Lb + j], -diff * inv);
  }
}

// g_kp = scale * R^T g_out   (keypoint_detector.py:182-184)
__global__ void transform_points_bwd_kernel(const float* __restrict__ g, const float* __restrict__ R,
                                            const float* __restrict__ scale, float* __restrict__ gk, int B, int M) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * M) return;
  int b = t / M, m = t - b * M;
  const float* r = R + (size_t)b * 9;
  const float s = scale[b];
  const float gx = g[(size_t)b * 3 * M + m] * s, gy = g[(size_t)b * 3 * M + M + m] * s, gz = g[(size_t)b * 3 * M + 2 * M + m] * s;
  for (int c = 0; c < 3; ++c) gk[(size_t)b * 3 * M + (size_t)c * M + m] = r[0 * 3 + c] * gx + r[1 * 3 + c] * gy + r[2 * 3 + c] * gz;
}

// ---- descriptor losses (models/losses.py:190-237, DescPairScanLoss) -----------------------------------------
// min_j || a[:, i] - b[:, j] ||_2 over C-dimensional descriptors, a (B,C,Ma), b (B,C,Nb) channel-major.
// CTA = (batch, 32 queries): the query tile lives in shared memory, database columns stream through a second tile.
constexpr int DP_Q = 32, DP_J = 64;
__global__ void __launch_bounds__(256)
desc_pairmin_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ min_d,
                    int32_t* __restrict__ arg, int C, int Ma, int Nb) {
  extern __shared__ float sm[];                  // [C][DP_Q] queries, then [C][DP_J] database tile
  float* sa = sm; float* sb = sm + (size_t)C * DP_Q;
  __shared__ float rbest[8][DP_Q]; __shared__ int rarg[8][DP_Q];
  const int bb = blockIdx.y, i0 = blockIdx.x * DP_Q;
  const int qi = threadIdx.x & 31, js = threadIdx.x >> 5;          // query, database slice (8 slices of 8 columns)
  const float* pa = a + (size_t)bb * C * Ma; const float* pb = b + (size_t)bb * C * Nb;
  for (int t = threadIdx.x; t < C * DP_Q; t += 256) { int c = t / DP_Q, q = t - c * DP_Q; sa[t] = (i0 + q) < Ma ? pa[(size_t)c * Ma + i0 + q] : 0.f; }
  float best = INFINITY; int bj = 0;
  for (int j0 = 0; j0 < Nb; j0 += DP_J) {
    __syncthreads();
    for (int t = threadIdx.x; t < C * DP_J; t += 256) { int c = t / DP_J, j = t - c * DP_J; sb[t] = (j0 + j) < Nb ? pb[(size_t)c * Nb + j0 + j] : 0.f; }
    __syncthreads();
    float acc[8];
    desc_sqdist_tile<8>(sa + qi, DP_Q, sb + js * 8, DP_J, C, acc);
#pragma unroll
    for (int u = 0; u < 8; ++u) { const int j = j0 + js * 8 + u; if (j < Nb && acc[u] < best) { best = acc[u]; bj = j; } }
  }
  rbest[js][qi] = best; rarg[js][qi] = bj;
  __syncthreads();
  if (threadIdx.x < DP_Q && i0 + threadIdx.x < Ma) {
    float bst = INFINITY; int bjj = 0;
    for (int t = 0; t < 8; ++t) { float v = rbest[t][threadIdx.x]; int j = rarg[t][threadIdx.x]; if (v < bst || (v == bst && j < bjj)) { bst = v; bjj = j; } }
    min_d[(size_t)bb * Ma + i0 + threadIdx.x] = sqrtf(bst);
    if (arg) arg[(size_t)bb * Ma + i0 + threadIdx.x] = bjj;
  }
}

// loss[b,m] = w[b,m] * max(dpos - dneg + gamma, 0), w = clamp(sigma_max - sigma, 0) / mean_m(...); active[b] = mean(dpos-dneg+gamma > 0)
__global__ void __launch_bounds__(256)
desc_triplet_kernel(const float* __restrict__ dpos, const float* __restrict__ dneg, const float* __restrict__ sigma,
                    float gamma, float sigma_max, float* __restrict__ loss, float* __restrict__ active, int M) {
  __shared__ double sh[32];
  const int b = blockIdx.x;
  double wsum = 0.0, act = 0.0;
  for (int m = threadIdx.x; m < M; m += 256) {
    wsum += fmaxf(sigma_max - sigma[(size_t)b * M + m], 0.f);
    act += (dpos[(size_t)b * M + m] - dneg[(size_t)b * M + m] + gamma) > 0.f ? 1.0 : 0.0;
  }
  __shared__ float wmean;
  double r = block_sum(wsum, sh);
  if (threadIdx.x == 0) wmean = (float)(r / M);
  r = block_sum(act, sh);
  if (threadIdx.x == 0) active[b] = (float)(r / M);
  __syncthreads();
  for (int m = threadIdx.x; m < M; m += 256) {
    const float w = fmaxf(sigma_max - sigma[(size_t)b * M + m], 0.f) / wmean;
    loss[(size_t)b * M + m] = w * fmaxf(dpos[(size_t)b * M + m] - dneg[(size_t)b * M + m] + gamma, 0.f);
  }
}


// PointOnSurfaceLoss (losses.py:146-183) after the nearest-point search: p = pc[:, arg], n = sn[0:3, arg],
//   u = (kp - p) / (||kp - p|| + 1e-7),  loss = (n . u)^2     (B,M); the arg-min is not differentiated.
// backward (g given): d = kp - p, r = ||d||, e = r + 1e-7, s = n . u:
//   dloss/dkp = 2 s * ( n / e - d * (n . d) / (r * e^2) )     (r = 0: torch.norm's sub-gradient is 0 -> only n / e, and s = 0)
__global__ void point_on_surface_kernel(const float* __restrict__ kp, const float* __restrict__ pc, const float* __restrict__ sn,
                                        const int32_t* __restrict__ arg, const float* __restrict__ g, float* __restrict__ loss,
                                        float* __restrict__ g_kp, int B, int M, int N, int S) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * M) return;
  const int b = t / M, m = t - b * M;
  const int j = arg[t];
  const float* k = kp + (size_t)b * 3 * M; const float* p = pc + (size_t)b * 3 * N; const float* n = sn + (size_t)b * S * N;
  const float dx = k[m] - p[j], dy = k[M + m] - p[N + j], dz = k[2 * M + m] - p[2 * N + j];
  const float nx = n[j], ny = n[N + j], nz = n[2 * N + j];
  const float r = sqrtf(dx * dx + dy * dy + dz * dz), e = r + 1e-7f;
  const float ux = dx / e, uy = dy / e, uz = dz / e;
  const float s = nx * ux + ny * uy + nz * uz;
  if (loss) loss[t] = s * s;
  if (g_kp) {
    const float nd = nx * dx + ny * dy + nz * dz;
    const float c = r > 0.f ? nd / (r * e * e) : 0.f;
    const float f = 2.f * s * g[t];
    float* o = g_kp + (size_t)b * 3 * M;
    o[m] = f * (nx / e - dx * c); o[M + m] = f * (ny / e - dy * c); o[2 * M + m] = f * (nz / e - dz * c);
  }
}

}  // namespace usip

using namespace usip;

extern "C" int usip_pairwise_min_f32(const float* a, const float* b, float* min_d, int32_t* arg,
                                     unsigned long long* packed, int B, int Ma, int Nb, void* stream) {
  USIP_REQUIRE(a && b && packed && B > 0 && Ma > 0 && Nb > 0, "pairwise_min: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  if (Nb <= 4 * PM_TILE) {
    pairwise_min_direct_kernel<128><<<dim3(cdiv(Ma, 128), B), PM_THREADS, 0, st>>>(a, b, min_d, arg, Ma, Nb);
    return check_launch("pairwise_min_direct_kernel");
  }
  size_t n = (size_t)B * Ma;
  pm_init_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, st>>>(packed, n);
  dim3 grid(cdiv(Nb, PM_TILE), cdiv(Ma, PM_Q), B);
  pairwise_min_kernel<<<grid, PM_THREADS, 0, st>>>(a, b, packed, Ma, Nb);
  pm_finish_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, st>>>(packed, min_d, arg, n);
  return check_launch("pairwise_min");
}

extern "C" int usip_chamfer_prob_reduce(const float* d_sd, const int32_t* i_sd, const float* d_ds,
                                        const int32_t* i_ds, const float* sig_src, const float* sig_dst,
                                        float* out3, int B, int M, int N, void* stream) {
  USIP_REQUIRE(d_sd && i_sd && d_ds && i_ds && sig_src && sig_dst && out3, "chamfer_prob_reduce: bad args");
  chamfer_prob_reduce_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(d_sd, i_sd, d_ds, i_ds, sig_src, sig_dst, out3,
                                                                  B, M, N);
  return check_launch("chamfer_prob_reduce_kernel");
}

extern "C" int usip_transform_points(const float* kp, const float* R, const float* scale, const float* shift,
                                     float* out, int B, int M, void* stream) {
  USIP_REQUIRE(kp && R && scale && shift && out, "transform_points: bad args");
  transform_points_kernel<<<cdiv(B * M, 256), 256, 0, (cudaStream_t)stream>>>(kp, R, scale, shift, out, B, M);
  return check_launch("transform_points_kernel");
}

extern "C" int usip_mean_scale(const float* d, int64_t n, float alpha, float* out, void* stream) {
  USIP_REQUIRE(d && out && n > 0, "mean_scale: bad args");
  mean_scale_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(d, n, alpha, out);
  return check_launch("mean_scale_kernel");
}

extern "C" int usip_pairwise_min_bwd(const float* a, const float* b, const float* min_d, const int32_t* arg,
                                     const float* g, float gscale, float* grad_a, float* grad_b, int B, int Ma,
                                     int Nb, void* stream) {
  USIP_REQUIRE(a && b && min_d && arg, "pairwise_min_bwd: bad args");
  pairwise_min_bwd_kernel<<<cdiv(B * Ma, 256), 256, 0, (cudaStream_t)stream>>>(a, b, min_d, arg, g, gscale, grad_a,
                                                                             grad_b, B, Ma, Nb);
  return check_launch("pairwise_min_bwd_kernel");
}

extern "C" int usip_chamfer_prob_bwd(const float* src, const float* dst, const float* sig_src, const float* sig_dst,
                                     const float* d_sd, const int32_t* i_sd, const float* d_ds, const int32_t* i_ds,
                                     const float* gout, float* g_src, float* g_dst, float* g_sig_src,
                                     float* g_sig_dst, int B, int M, int N, void* stream) {
  USIP_REQUIRE(src && dst && sig_src && sig_dst && gout && g_src && g_dst && g_sig_src && g_sig_dst,
               "chamfer_prob_bwd: bad args");
  chamfer_prob_bwd_kernel<<<cdiv(B * (M + N), 256), 256, 0, (cudaStream_t)stream>>>(
      src, dst, sig_src, sig_dst, d_sd, i_sd, d_ds, i_ds, gout, g_src, g_dst, g_sig_src, g_sig_dst, B, M, N);
  return check_launch("chamfer_prob_bwd_kernel");
}

extern "C" int usip_transform_points_bwd(const float* g_out, const float* R, const float* scale, float* g_kp,
                                         int B, int M, void* stream) {
  USIP_REQUIRE(g_out && R && scale && g_kp, "transform_points_bwd: bad args");
  transform_points_bwd_kernel<<<cdiv(B * M, 256), 256, 0, (cudaStream_t)stream>>>(g_out, R, scale, g_kp, B, M);
  return check_launch("transform_points_bwd_kernel");
}

extern "C" int usip_desc_pairmin_f32(const float* a, const float* b, float* min_d, int32_t* arg, int B, int C, int Ma,
                                     int Nb, void* stream) {
  USIP_REQUIRE(a && b && min_d && B > 0 && C > 0 && Ma > 0 && Nb > 0, "desc_pairmin: bad args");
  size_t smem = (size_t)C * (DP_Q + DP_J) * sizeof(float);
  USIP_REQUIRE(smem <= 200 * 1024, "desc_pairmin: C too large");
  if (smem > 40 * 1024) cudaFuncSetAttribute(desc_pairmin_kernel   /* + 2 KB static */, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  dim3 grid(cdiv(Ma, DP_Q), B);
  desc_pairmin_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(a, b, min_d, arg, C, Ma, Nb);
  return check_launch("desc_pairmin_kernel");
}

extern "C" int usip_desc_triplet(const float* dpos, const float* dneg, const float* sigma, float gamma, float sigma_max,
                                 float* loss, float* active, int B, int M, void* stream) {
  USIP_REQUIRE(dpos && dneg && sigma && loss && active, "desc_triplet: bad args");
  desc_triplet_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(dpos, dneg, sigma, gamma, sigma_max, loss, active, M);
  return check_launch("desc_triplet_kernel");
}

extern "C" int usip_point_on_surface(const float* kp, const float* pc, const float* sn, const int32_t* arg, const float* g,
                                     float* loss, float* g_kp, int B, int M, int N, int S, void* stream) {
  USIP_REQUIRE(kp && pc && sn && arg && (loss || (g && g_kp)) && S >= 3, "point_on_surface: bad args");
  point_on_surface_kernel<<<cdiv(B * M, 256), 256, 0, (cudaStream_t)stream>>>(kp, pc, sn, arg, g, loss, g_kp, B, M, N, S);
  return check_launch("point_on_surface_kernel");
}
