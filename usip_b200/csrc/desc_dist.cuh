// desc_dist.cuh -- the squared descriptor distance shared by the nearest-descriptor searches (usip_desc_pairmin_f32 in
// loss.cu, usip_desc_knn_f32 in registration.cu).  One formula, so the k = 1 column of the kNN search is bit-identical
// to the loss's arg-min: an fmaf chain over the channels in ascending order, df = a - b, acc = fmaf(df, df, acc).
#pragma once

namespace usip {

// acc[u] = sum_c (qa[c * lda] - tb[c * ldb + u])^2 for u < U: one query column against U database columns, both in
// channel-major tiles (shared memory in both callers).
template <int U>
__device__ __forceinline__ void desc_sqdist_tile(const float* qa, int lda, const float* tb, int ldb, int C, float (&acc)[U]) {
#pragma unroll
  for (int u = 0; u < U; ++u) acc[u] = 0.f;
  for (int c = 0; c < C; ++c) {
    const float av = qa[c * lda];
#pragma unroll
    for (int u = 0; u < U; ++u) { const float df = av - tb[c * ldb + u]; acc[u] = fmaf(df, df, acc[u]); }
  }
}

}  // namespace usip
