// registration.cu -- registration evaluation of a trained detector + descriptor (the paper's success rate, RTE / RRE):
// k-nearest descriptor matching, the correspondence list, and a batched RANSAC rigid fit.
// Restates evaluation/matlab/eval_outdoor/{kitti/evaluate_kitti.m, oxford/evaluate_oxford.m} and
// eval_outdoor/external/{ransacfitRt,ransac,estimateRt,estimateRigidTransform,quat2rot,crossTimesMatrix}.m.
//
// This file is compiled with -fmad=false (build.py): no multiply-add is contracted, so the float64 3-point fit gives the
// same bits in the scoring kernel and in the refit kernel that re-derives the winning hypothesis.  The residual below also
// spells its rounding out (__dmul_rn / __dadd_rn), as the oracle restates it.
#include "common.cuh"
#include "desc_dist.cuh"
#include <float.h>
#include <curand_philox4x32_x.h>

namespace usip {

// ---- 1. k nearest descriptors  (pdist2(pos_desc, anc_desc, 'euclidean', 'smallest', k), evaluate_kitti.m:53) --------
// CTA = (pair, 32 queries), 8 warps = 8 slices of 8 columns of every 64-column database tile (the layout of
// desc_pairmin_kernel, loss.cu).  Each thread keeps a sorted top-K of its columns (ascending j, strict '<': the earlier
// index stays first on ties); the 8 slice lists of a query are merged by (distance, index).
constexpr int KN_Q = 32, KN_J = 64;

template <int K>
__global__ void __launch_bounds__(256)
desc_knn_kernel(const float* __restrict__ a, const float* __restrict__ b, const int32_t* __restrict__ na,
                const int32_t* __restrict__ nb, int32_t* __restrict__ idx, float* __restrict__ dist, int C, int Ma, int Mb) {
  extern __shared__ float sm[];                  // [C][KN_Q] queries, then [C][KN_J] database tile
  float* sa = sm; float* sb = sm + (size_t)C * KN_Q;
  __shared__ float rd[8][K][KN_Q]; __shared__ int ri[8][K][KN_Q];
  const int bb = blockIdx.y, i0 = blockIdx.x * KN_Q;
  const int qi = threadIdx.x & 31, js = threadIdx.x >> 5;
  const int nq = na ? min(na[bb], Ma) : Ma, nd = nb ? min(nb[bb], Mb) : Mb;
  const float* pa = a + (size_t)bb * C * Ma; const float* pb = b + (size_t)bb * C * Mb;
  for (int t = threadIdx.x; t < C * KN_Q; t += 256) { int c = t / KN_Q, q = t - c * KN_Q; sa[t] = (i0 + q) < nq ? pa[(size_t)c * Ma + i0 + q] : 0.f; }
  float bd[K]; int bi[K];
#pragma unroll
  for (int s = 0; s < K; ++s) { bd[s] = INFINITY; bi[s] = -1; }
  for (int j0 = 0; j0 < nd; j0 += KN_J) {
    __syncthreads();
    for (int t = threadIdx.x; t < C * KN_J; t += 256) { int c = t / KN_J, j = t - c * KN_J; sb[t] = (j0 + j) < nd ? pb[(size_t)c * Mb + j0 + j] : 0.f; }
    __syncthreads();
    float acc[8];
    desc_sqdist_tile<8>(sa + qi, KN_Q, sb + js * 8, KN_J, C, acc);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const int j = j0 + js * 8 + u; const float d = acc[u];
      if (j < nd && d < bd[K - 1]) {             // insertion from the back; every bd[s] read below is still the old one
#pragma unroll
        for (int s = K - 1; s > 0; --s) {
          if (d < bd[s - 1]) { bd[s] = bd[s - 1]; bi[s] = bi[s - 1]; }
          else if (d < bd[s]) { bd[s] = d; bi[s] = j; }
        }
        if (d < bd[0]) { bd[0] = d; bi[0] = j; }
      }
    }
  }
#pragma unroll
  for (int s = 0; s < K; ++s) { rd[js][s][qi] = bd[s]; ri[js][s][qi] = bi[s]; }
  __syncthreads();
  const int i = i0 + threadIdx.x;
  if (threadIdx.x >= KN_Q || i >= Ma) return;
  int32_t* oi = idx + ((size_t)bb * Ma + i) * K;
  float* od = dist ? dist + ((size_t)bb * Ma + i) * K : nullptr;
  int h[8];
#pragma unroll
  for (int s = 0; s < 8; ++s) h[s] = 0;
  for (int r = 0; r < K; ++r) {
    float best = INFINITY; int bj = -1, bs = -1;
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      if (h[s] < K) {
        const float v = rd[s][h[s]][threadIdx.x]; const int j = ri[s][h[s]][threadIdx.x];
        if (j >= 0 && (bj < 0 || v < best || (v == best && j < bj))) { best = v; bj = j; bs = s; }
      }
    }
#pragma unroll
    for (int s = 0; s < 8; ++s) h[s] += (s == bs);
    const bool ok = i < nq && bj >= 0;
    oi[r] = ok ? bj : -1;
    if (od) od[r] = ok ? sqrtf(best) : INFINITY;
  }
}

// ---- 2. correspondence list  (evaluate_kitti.m:53-54; evaluate_oxford.m:63-72, union(..., 'rows')) --------------------
// One CTA per pair: every (anc, pos) match sets a bit of an Ma x Mb bitmap in shared memory, and an ordered compaction
// (each thread owns a contiguous run of words, block exclusive scan of the popcounts) emits the set bits in row-major
// order -- the unique rows in ascending (anc, pos) order that union() returns.  With k = 1 and one direction, row i holds
// the single bit nn(i), so the list is [i, nn(i)] in anc order, as evaluate_kitti.m builds it.
__global__ void __launch_bounds__(1024)
corr_build_kernel(const int32_t* __restrict__ nn12, int k12, const int32_t* __restrict__ nn21, int k21,
                  const int32_t* __restrict__ na, const int32_t* __restrict__ nb, int Ma, int Mb,
                  int32_t* __restrict__ corr, int32_t* __restrict__ count, int nmax) {
  extern __shared__ uint32_t bits[];             // [Ma][W]
  __shared__ int wtot[32];
  __shared__ int total;
  const int b = blockIdx.x, W = (Mb + 31) >> 5, nw = Ma * W;
  const int nq = na ? min(na[b], Ma) : Ma, nd = nb ? min(nb[b], Mb) : Mb;
  for (int t = threadIdx.x; t < nw; t += blockDim.x) bits[t] = 0u;
  __syncthreads();
  for (int t = threadIdx.x; t < nq * k12; t += blockDim.x) {
    const int i = t / k12, j = nn12[((size_t)b * Ma + i) * k12 + (t - i * k12)];
    if (j >= 0 && j < nd) atomicOr(&bits[i * W + (j >> 5)], 1u << (j & 31));
  }
  if (nn21)
    for (int t = threadIdx.x; t < nd * k21; t += blockDim.x) {
      const int j = t / k21, i = nn21[((size_t)b * Mb + j) * k21 + (t - j * k21)];
      if (i >= 0 && i < nq) atomicOr(&bits[i * W + (j >> 5)], 1u << (j & 31));
    }
  __syncthreads();
  const int per = (nw + blockDim.x - 1) / blockDim.x;
  const int w0 = min(nw, (int)threadIdx.x * per), w1 = min(nw, w0 + per);
  int c = 0;
  for (int w = w0; w < w1; ++w) c += __popc(bits[w]);
  const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
  int inc = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
  if (lane == 31) wtot[wp] = inc;
  __syncthreads();
  if (wp == 0) {
    const int nwarps = blockDim.x >> 5;
    int v = lane < nwarps ? wtot[lane] : 0, s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += u; }
    if (lane < nwarps) wtot[lane] = s - v;       // exclusive
    if (lane == 31) total = s;
  }
  __syncthreads();
  int o = wtot[wp] + inc - c;
  int32_t* out = corr + (size_t)b * nmax * 2;
  for (int w = w0; w < w1; ++w) {
    uint32_t m = bits[w];
    const int i = w / W, jb = (w - i * W) << 5;
    while (m) {
      const int j = jb + __ffs(m) - 1; m &= m - 1;
      out[2 * o] = i; out[2 * o + 1] = j; ++o;
    }
  }
  for (int t = total + threadIdx.x; t < nmax; t += blockDim.x) { out[2 * t] = -1; out[2 * t + 1] = -1; }
  if (threadIdx.x == 0) count[b] = total;
}

// ---- 3. rigid fit  (estimateRigidTransform.m, quat2rot.m, crossTimesMatrix.m) --------------------------------------
struct Rigid { double r[9]; double t[3]; };      // x = R y + t: pos-frame points into the anc frame

// B += A^T A with A = [0, (y-x)^T ; (x-y), [y+x]_x] for one centred pair (estimateRigidTransform.m:51-61, crossTimesMatrix.m:18-26); upper
// triangle of the symmetric 4x4 B, row-major: 00 01 02 03 11 12 13 22 23 33.
__device__ __forceinline__ void taati_accumulate(double (&Bm)[10], const double (&x)[3], const double (&y)[3]) {
  const double d0 = y[0] - x[0], d1 = y[1] - x[1], d2 = y[2] - x[2];
  const double s0 = y[0] + x[0], s1 = y[1] + x[1], s2 = y[2] + x[2];
  const double A[4][4] = {{0.0, d0, d1, d2}, {-d0, 0.0, -s2, s1}, {-d1, s2, 0.0, -s0}, {-d2, -s1, s0, 0.0}};
  int k = 0;
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = p; q < 4; ++q, ++k) Bm[k] = Bm[k] + (((A[0][p] * A[0][q] + A[1][p] * A[1][q]) + A[2][p] * A[2][q]) + A[3][p] * A[3][q]);
}

template <int P, int Q>
__device__ __forceinline__ void jacobi_rotate(double (&a)[4][4], double (&v)[4][4]) {
  const double apq = a[P][Q];
  if (apq == 0.0) return;
  const double theta = (a[Q][Q] - a[P][P]) / (2.0 * apq);
  const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
  const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
  for (int k = 0; k < 4; ++k) { const double kp = a[k][P], kq = a[k][Q]; a[k][P] = c * kp - s * kq; a[k][Q] = s * kp + c * kq; }
#pragma unroll
  for (int k = 0; k < 4; ++k) { const double pk = a[P][k], qk = a[Q][k]; a[P][k] = c * pk - s * qk; a[Q][k] = s * pk + c * qk; }
#pragma unroll
  for (int k = 0; k < 4; ++k) { const double kp = v[k][P], kq = v[k][Q]; v[k][P] = c * kp - s * kq; v[k][Q] = s * kp + c * kq; }
}

// The quaternion is B's eigenvector of the smallest eigenvalue (the last right-singular vector of the symmetric PSD B,
// estimateRigidTransform.m:63-64): cyclic Jacobi until the off-diagonal mass is below double rounding, then the column
// of the smallest diagonal entry (first on ties).  quat2rot.m:15-25 (w first) and t = x_c - R y_c (estimateRigidTransform.m:67-71).
__device__ __forceinline__ void rigid_from_B(const double (&Bm)[10], const double (&xc)[3], const double (&yc)[3], Rigid& m) {
  double a[4][4], v[4][4];
  int k = 0;
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = p; q < 4; ++q, ++k) { a[p][q] = Bm[k]; a[q][p] = Bm[k]; }
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) v[p][q] = p == q ? 1.0 : 0.0;
#pragma unroll 1
  for (int sweep = 0; sweep < 16; ++sweep) {
    const double off = ((((a[0][1] * a[0][1] + a[0][2] * a[0][2]) + a[0][3] * a[0][3]) + a[1][2] * a[1][2]) + a[1][3] * a[1][3]) + a[2][3] * a[2][3];
    const double dg = ((a[0][0] * a[0][0] + a[1][1] * a[1][1]) + a[2][2] * a[2][2]) + a[3][3] * a[3][3];
    if (!(off > 1e-36 * dg)) break;
    jacobi_rotate<0, 1>(a, v); jacobi_rotate<0, 2>(a, v); jacobi_rotate<0, 3>(a, v);
    jacobi_rotate<1, 2>(a, v); jacobi_rotate<1, 3>(a, v); jacobi_rotate<2, 3>(a, v);
  }
  double best = a[0][0], q0 = v[0][0], q1 = v[1][0], q2 = v[2][0], q3 = v[3][0];
#pragma unroll
  for (int c = 1; c < 4; ++c)
    if (a[c][c] < best) { best = a[c][c]; q0 = v[0][c]; q1 = v[1][c]; q2 = v[2][c]; q3 = v[3][c]; }
  double* R = m.r;
  R[0] = q0 * q0 + q1 * q1 - q2 * q2 - q3 * q3; R[1] = 2.0 * (q1 * q2 - q0 * q3);                R[2] = 2.0 * (q1 * q3 + q0 * q2);
  R[3] = 2.0 * (q1 * q2 + q0 * q3);                R[4] = q0 * q0 - q1 * q1 + q2 * q2 - q3 * q3; R[5] = 2.0 * (q2 * q3 - q0 * q1);
  R[6] = 2.0 * (q1 * q3 - q0 * q2);                R[7] = 2.0 * (q2 * q3 + q0 * q1);                R[8] = q0 * q0 - q1 * q1 - q2 * q2 + q3 * q3;
#pragma unroll
  for (int r = 0; r < 3; ++r) m.t[r] = xc[r] - ((R[3 * r] * yc[0] + R[3 * r + 1] * yc[1]) + R[3 * r + 2] * yc[2]);
}

__device__ __forceinline__ void load_corr(const double* anc, const double* pos, const int32_t* cr, int c, double (&x)[3], double (&y)[3]) {
  const double* pa = anc + (size_t)cr[2 * c] * 3; const double* pp = pos + (size_t)cr[2 * c + 1] * 3;
  x[0] = pa[0]; x[1] = pa[1]; x[2] = pa[2]; y[0] = pp[0]; y[1] = pp[1]; y[2] = pp[2];
}

// estimateRt.m on the three sampled correspondences (centroids summed in index order, as sum(x, 2) does; estimateRigidTransform.m:45-46)
__device__ __forceinline__ void fit3(const double* anc, const double* pos, const int32_t* cr, int i0, int i1, int i2, Rigid& m) {
  double x[3][3], y[3][3];
  load_corr(anc, pos, cr, i0, x[0], y[0]); load_corr(anc, pos, cr, i1, x[1], y[1]); load_corr(anc, pos, cr, i2, x[2], y[2]);
  double xc[3], yc[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) { xc[r] = ((x[0][r] + x[1][r]) + x[2][r]) / 3.0; yc[r] = ((y[0][r] + y[1][r]) + y[2][r]) / 3.0; }
  double Bm[10];
#pragma unroll
  for (int k = 0; k < 10; ++k) Bm[k] = 0.0;
#pragma unroll
  for (int u = 0; u < 3; ++u) {
    const double xs[3] = {x[u][0] - xc[0], x[u][1] - xc[1], x[u][2] - xc[2]};
    const double ys[3] = {y[u][0] - yc[0], y[u][1] - yc[1], y[u][2] - yc[2]};
    taati_accumulate(Bm, xs, ys);
  }
  rigid_from_B(Bm, xc, yc, m);
}

// ||x - (R y + t)|| (ransacfitRt.m:73-74), every operation rounded in this order: p_r = ((R_r0 y0 + R_r1 y1) + R_r2 y2) + t_r,
// d^2 = (dx^2 + dy^2) + dz^2, correctly rounded sqrt.
__device__ __forceinline__ double residual(const Rigid& m, const double (&x)[3], const double (&y)[3]) {
  double e[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double p = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(m.r[3 * r], y[0]), __dmul_rn(m.r[3 * r + 1], y[1])),
                                         __dmul_rn(m.r[3 * r + 2], y[2])), m.t[r]);
    e[r] = __dsub_rn(x[r], p);
  }
  return __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(e[0], e[0]), __dmul_rn(e[1], e[1])), __dmul_rn(e[2], e[2])));
}

// ---- 4. RANSAC  (ransac.m:140-218 with s = 3 and isdegenerate = 0: exactly one sample per trial) -------------------
// Trial tau of pair b: three distinct uniform indices in [0, n) from Philox-4x32-10 at counter (tau, b, 0, 0), key = seed.
// (u * m) >> 32 maps a 32-bit draw to [0, m); the 2nd draw skips the 1st index, the 3rd skips the smaller then the larger.
__device__ __forceinline__ void draw3(unsigned long long seed, int b, int tau, int n, int& i0, int& i1, int& i2) {
  const uint4 r = curand_Philox4x32_10(make_uint4((unsigned)tau, (unsigned)b, 0u, 0u),
                                       make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
  i0 = (int)(((unsigned long long)r.x * (unsigned)n) >> 32);
  i1 = (int)(((unsigned long long)r.y * (unsigned)(n - 1)) >> 32);
  if (i1 >= i0) ++i1;
  i2 = (int)(((unsigned long long)r.z * (unsigned)(n - 2)) >> 32);
  const int lo = min(i0, i1), hi = max(i0, i1);
  if (i2 >= lo) ++i2;
  if (i2 >= hi) ++i2;
}

__device__ __forceinline__ void trial_sample(const int32_t* samples, int32_t* samples_out, unsigned long long seed, int b, int tau,
                                             int T, int n, int& i0, int& i1, int& i2) {
  if (samples) {
    const int32_t* s = samples + ((size_t)b * T + tau) * 3; i0 = s[0]; i1 = s[1]; i2 = s[2];
  } else {
    draw3(seed, b, tau, n, i0, i1, i2);
  }
  if (samples_out) { int32_t* s = samples_out + ((size_t)b * T + tau) * 3; s[0] = i0; s[1] = i1; s[2] = i2; }
}

// Per-pair loop state: N (the adaptive trial bound), done; trialcount / bestscore / best_trial live in the outputs.
__global__ void ransac_init_kernel(const int32_t* __restrict__ ncorr, double* __restrict__ Nst, int32_t* __restrict__ done,
                                   int32_t* __restrict__ trialcount, int32_t* __restrict__ bestscore,
                                   int32_t* __restrict__ best_trial, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  Nst[b] = 1.0; trialcount[b] = 0; bestscore[b] = 0; best_trial[b] = -1;
  done[b] = ncorr[b] <= 3;                       // ransacfitRt.m:25-35: no loop for n < 3 (empty) or n == 3 (direct fit)
}

// One thread per hypothesis, 64 trials of one pair per CTA; the pair's correspondences stream through shared memory and
// every lane reads the same one (broadcast).  Writes only the inlier count of each trial.
constexpr int RS_THREADS = 64, RS_TILE = 128;
__global__ void __launch_bounds__(RS_THREADS)
ransac_score_kernel(const double* __restrict__ anc, const double* __restrict__ pos, const int32_t* __restrict__ corr,
                    const int32_t* __restrict__ ncorr, const int32_t* __restrict__ samples, int32_t* __restrict__ samples_out,
                    unsigned long long seed, double thr, const int32_t* __restrict__ done, int32_t* __restrict__ counts,
                    int T, int t0, int t1, int Ma, int Mb, int nmax) {
  __shared__ double sx[3][RS_TILE], sy[3][RS_TILE];
  const int b = blockIdx.y;
  const int base = t0 + blockIdx.x * RS_THREADS;
  if (base >= t1 || done[b]) return;             // uniform over the CTA
  const int n = ncorr[b];
  const double* pa = anc + (size_t)b * Ma * 3; const double* pp = pos + (size_t)b * Mb * 3;
  const int32_t* cr = corr + (size_t)b * nmax * 2;
  const int tau = base + threadIdx.x;
  const bool active = tau < t1;
  Rigid m;
  if (active) {
    int i0, i1, i2;
    trial_sample(samples, samples_out, seed, b, tau, T, n, i0, i1, i2);
    fit3(pa, pp, cr, i0, i1, i2, m);
  }
  int cnt = 0;
  for (int c0 = 0; c0 < n; c0 += RS_TILE) {
    const int cc = min(RS_TILE, n - c0);
    __syncthreads();
    for (int t = threadIdx.x; t < cc; t += RS_THREADS) {
      double x[3], y[3];
      load_corr(pa, pp, cr, c0 + t, x, y);
#pragma unroll
      for (int r = 0; r < 3; ++r) { sx[r][t] = x[r]; sy[r][t] = y[r]; }
    }
    __syncthreads();
    if (active)
      for (int t = 0; t < cc; ++t) {
        const double x[3] = {sx[0][t], sx[1][t], sx[2][t]}, y[3] = {sy[0][t], sy[1][t], sy[2][t]};
        cnt += residual(m, x, y) < thr;
      }
  }
  if (active) counts[(size_t)b * T + tau] = cnt;
}

// One thread per pair advances ransac.m:140-218 over trials [t0, t1) of the counts; pairs already terminated return.
__global__ void ransac_scan_kernel(const int32_t* __restrict__ counts, const int32_t* __restrict__ ncorr, int T, int t0, int t1,
                                   double p, int max_trials, double* __restrict__ Nst, int32_t* __restrict__ done,
                                   int32_t* __restrict__ trialcount, int32_t* __restrict__ bestscore,
                                   int32_t* __restrict__ best_trial, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B || done[b]) return;
  const double n = (double)ncorr[b], lp = log(1.0 - p);
  double N = Nst[b];
  int tc = trialcount[b], bs = bestscore[b], bt = best_trial[b];
  bool fin = false;
  for (int tau = t0; tau < t1; ++tau) {          // tc == tau here: trials are consumed in order
    if (!(N > (double)tc)) { fin = true; break; }                     // ransac.m:140
    const int ninl = counts[(size_t)b * T + tau];
    if (ninl >= bs) {                                                 // ransac.m:195, '>=': ties go to the later trial
      bs = ninl; bt = tau;
      const double f = (double)ninl / n;
      double pno = 1.0 - f * f * f;
      pno = fmin(1.0 - DBL_EPSILON, fmax(DBL_EPSILON, pno));
      N = fmax(lp / log(pno), 10.0);                                  // ransac.m:202-207 (f^3 as f*f*f)
    }
    if (++tc > max_trials) { fin = true; break; }
  }
  Nst[b] = N; trialcount[b] = tc; bestscore[b] = bs; best_trial[b] = bt; done[b] = fin;
}

// fixed-order block sum of V doubles (warp xor tree, then warps in index order); result valid on thread 0
template <int V>
__device__ __forceinline__ void block_sum_fixed(double (&v)[V], double (*sh)[V]) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < V; ++k) v[k] = warp_sum_d(v[k]);
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < V; ++k) sh[w][k] = v[k];
  __syncthreads();
  if (threadIdx.x == 0)
#pragma unroll
    for (int k = 0; k < V; ++k) { double s = sh[0][k]; for (int u = 1; u < (int)(blockDim.x >> 5); ++u) s += sh[u][k]; v[k] = s; }
  __syncthreads();
}

// ransacfitRt.m:25-50: one CTA per pair re-derives the best hypothesis, marks its inliers (the returned set: not
// recomputed after the refit), and fits Rt to them with fixed-order float64 sums.  n == 3: direct fit on all three.
constexpr int RF_THREADS = 256;
__global__ void __launch_bounds__(RF_THREADS)
ransac_refit_kernel(const double* __restrict__ anc, const double* __restrict__ pos, const int32_t* __restrict__ corr,
                    const int32_t* __restrict__ ncorr, const int32_t* __restrict__ samples, unsigned long long seed, double thr,
                    const int32_t* __restrict__ best_trial, int32_t* __restrict__ n_inliers, double* __restrict__ Rt,
                    uint8_t* __restrict__ mask, int32_t* __restrict__ status, int T, int Ma, int Mb, int nmax) {
  __shared__ double sh[RF_THREADS / 32][10];
  __shared__ double cen[6];
  const int b = blockIdx.x, n = ncorr[b];
  const bool all = n == 3;
  const bool empty = n < 3 || (!all && n_inliers[b] < 3);
  uint8_t* mk = mask + (size_t)b * nmax;
  double* out = Rt + (size_t)b * 12;
  if (empty) {                                   // uniform over the CTA
    for (int c = threadIdx.x; c < nmax; c += RF_THREADS) mk[c] = 0;
    if (threadIdx.x < 12) out[threadIdx.x] = __longlong_as_double(0x7ff8000000000000ll);
    if (threadIdx.x == 0) { n_inliers[b] = 0; status[b] = n < 3 ? 1 : 2; }
    return;
  }
  const double* pa = anc + (size_t)b * Ma * 3; const double* pp = pos + (size_t)b * Mb * 3;
  const int32_t* cr = corr + (size_t)b * nmax * 2;
  Rigid h;
  if (!all) {
    int i0, i1, i2;
    trial_sample(samples, nullptr, seed, b, best_trial[b], T, n, i0, i1, i2);
    fit3(pa, pp, cr, i0, i1, i2, h);
  }
  double s[7] = {0, 0, 0, 0, 0, 0, 0};           // sum x, sum y, count
  for (int c = threadIdx.x; c < nmax; c += RF_THREADS) {
    bool in = false;
    if (c < n) {
      double x[3], y[3];
      load_corr(pa, pp, cr, c, x, y);
      in = all || residual(h, x, y) < thr;
      if (in) { s[0] += x[0]; s[1] += x[1]; s[2] += x[2]; s[3] += y[0]; s[4] += y[1]; s[5] += y[2]; s[6] += 1.0; }
    }
    mk[c] = in;
  }
  block_sum_fixed<7>(s, (double (*)[7])&sh[0][0]);
  if (threadIdx.x == 0)
#pragma unroll
    for (int k = 0; k < 6; ++k) cen[k] = s[k] / s[6];
  __syncthreads();
  const double cnt = s[6];                       // valid on thread 0
  const double xc[3] = {cen[0], cen[1], cen[2]}, yc[3] = {cen[3], cen[4], cen[5]};
  double Bm[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int c = threadIdx.x; c < n; c += RF_THREADS) {
    if (!mk[c]) continue;
    double x[3], y[3];
    load_corr(pa, pp, cr, c, x, y);
    const double xs[3] = {x[0] - xc[0], x[1] - xc[1], x[2] - xc[2]}, ys[3] = {y[0] - yc[0], y[1] - yc[1], y[2] - yc[2]};
    taati_accumulate(Bm, xs, ys);
  }
  block_sum_fixed<10>(Bm, sh);
  if (threadIdx.x == 0) {
    Rigid m;
    rigid_from_B(Bm, xc, yc, m);
#pragma unroll
    for (int r = 0; r < 3; ++r) { out[4 * r] = m.r[3 * r]; out[4 * r + 1] = m.r[3 * r + 1]; out[4 * r + 2] = m.r[3 * r + 2]; out[4 * r + 3] = m.t[r]; }
    n_inliers[b] = (int)cnt; status[b] = 0;
  }
}

// trial chunk ends of the termination scan: a pair that stops inside a chunk wastes at most the rest of that chunk
constexpr int RANSAC_CHUNKS = 5;
constexpr int RANSAC_CHUNK_ENDS[RANSAC_CHUNKS - 1] = {64, 320, 1344, 5440};

}  // namespace usip

using namespace usip;

extern "C" int usip_desc_knn_f32(const float* a, const float* b, const int32_t* na, const int32_t* nb, int32_t* idx, float* dist,
                                 int B, int C, int Ma, int Mb, int k, void* stream) {
  USIP_REQUIRE(a && b && idx && B > 0 && B <= 65535 && C > 0 && Ma > 0 && Mb > 0, "desc_knn: bad args");
  USIP_REQUIRE(k >= 1 && k <= 8, "desc_knn: k must be in [1, 8]");
  const size_t smem = (size_t)C * (KN_Q + KN_J) * sizeof(float);
  USIP_REQUIRE(smem <= 160 * 1024, "desc_knn: C too large (at most 426 channels)");
  const dim3 grid(cdiv(Ma, KN_Q), B);
  cudaStream_t st = (cudaStream_t)stream;
#define USIP_KNN_CASE(K)                                                                                               \
  case K:                                                                                                              \
    if (smem > 40 * 1024) cudaFuncSetAttribute(desc_knn_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    desc_knn_kernel<K><<<grid, 256, smem, st>>>(a, b, na, nb, idx, dist, C, Ma, Mb);                                   \
    break;
  switch (k) { USIP_KNN_CASE(1) USIP_KNN_CASE(2) USIP_KNN_CASE(3) USIP_KNN_CASE(4) USIP_KNN_CASE(5) USIP_KNN_CASE(6)
               USIP_KNN_CASE(7) USIP_KNN_CASE(8) }
#undef USIP_KNN_CASE
  return check_launch("desc_knn_kernel");
}

extern "C" int usip_corr_build(const int32_t* nn12, int k12, const int32_t* nn21, int k21, const int32_t* na, const int32_t* nb,
                               int32_t* corr, int32_t* count, int B, int Ma, int Mb, int nmax, void* stream) {
  USIP_REQUIRE(nn12 && corr && count && B > 0 && Ma > 0 && Mb > 0 && k12 >= 1 && (!nn21 || k21 >= 1), "corr_build: bad args");
  USIP_REQUIRE(Ma <= 1024 && Mb <= 1024, "corr_build: at most 1024 keypoints per frame (the Ma x Mb bitmap lives in shared memory)");
  const long long most = (long long)Ma * k12 + (nn21 ? (long long)Mb * k21 : 0);
  USIP_REQUIRE(nmax >= (int)min(most, (long long)Ma * Mb), "corr_build: nmax below the largest possible list");
  const size_t smem = (size_t)Ma * ((Mb + 31) / 32) * sizeof(uint32_t);
  if (smem > 40 * 1024) cudaFuncSetAttribute(corr_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  corr_build_kernel<<<B, 1024, smem, (cudaStream_t)stream>>>(nn12, k12, nn21, k21, na, nb, Ma, Mb, corr, count, nmax);
  return check_launch("corr_build_kernel");
}

extern "C" size_t usip_ransac_rt_scratch_bytes(int B, int max_trials) {
  return (size_t)B * sizeof(double) + (size_t)B * sizeof(int32_t) + (size_t)B * (max_trials + 1) * sizeof(int32_t) + 16;
}

extern "C" int usip_ransac_rt(const double* anc_xyz, const double* pos_xyz, const int32_t* corr, const int32_t* ncorr,
                              const int32_t* samples, int32_t* samples_out, double threshold, int max_trials, double p,
                              unsigned long long seed, double* Rt, int32_t* n_inliers, int32_t* trialcount, int32_t* best_trial,
                              uint8_t* inlier_mask, int32_t* status, void* scratch, size_t scratch_bytes, int B, int Ma, int Mb,
                              int nmax, void* stream) {
  USIP_REQUIRE(anc_xyz && pos_xyz && corr && ncorr && Rt && n_inliers && trialcount && best_trial && inlier_mask && status,
               "ransac_rt: bad args");
  USIP_REQUIRE(B > 0 && B <= 65535 && Ma > 0 && Mb > 0 && nmax > 0 && max_trials >= 0 && p > 0.0 && p < 1.0, "ransac_rt: bad sizes");
  USIP_REQUIRE(scratch && ((uintptr_t)scratch & 15) == 0 && scratch_bytes >= usip_ransac_rt_scratch_bytes(B, max_trials),
               "ransac_rt: scratch too small or misaligned");
  const int T = max_trials + 1;                  // trialcount stops at max_trials + 1 (ransac.m:216)
  double* Nst = (double*)scratch;
  int32_t* done = (int32_t*)(Nst + B);
  int32_t* counts = done + B;
  cudaStream_t st = (cudaStream_t)stream;
  ransac_init_kernel<<<cdiv(B, 128), 128, 0, st>>>(ncorr, Nst, done, trialcount, n_inliers, best_trial, B);
  // every chunk launches (possibly empty) so the launch count does not depend on max_trials
  for (int c = 0; c < RANSAC_CHUNKS; ++c) {
    const int t0 = c == 0 ? 0 : min(RANSAC_CHUNK_ENDS[c - 1], T);
    const int t1 = c == RANSAC_CHUNKS - 1 ? T : min(RANSAC_CHUNK_ENDS[c], T);
    ransac_score_kernel<<<dim3(max(1, cdiv(t1 - t0, RS_THREADS)), B), RS_THREADS, 0, st>>>(
        anc_xyz, pos_xyz, corr, ncorr, samples, samples_out, seed, threshold, done, counts, T, t0, t1, Ma, Mb, nmax);
    ransac_scan_kernel<<<cdiv(B, 128), 128, 0, st>>>(counts, ncorr, T, t0, t1, p, max_trials, Nst, done, trialcount, n_inliers,
                                                     best_trial, B);
  }
  ransac_refit_kernel<<<B, RF_THREADS, 0, st>>>(anc_xyz, pos_xyz, corr, ncorr, samples, seed, threshold, best_trial, n_inliers,
                                                Rt, inlier_mask, status, T, Ma, Mb, nmax);
  return check_launch("ransac_rt");
}
