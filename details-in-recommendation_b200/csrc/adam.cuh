// [TF] Adam._apply_sparse_shared as a sweep of a [T | m | v] table in tiles of kAdamTile rows: the scalar arithmetic
// and the tile body shared by dir_rows_apply_adam (adam.cu, one GPU) and dir_shard_owner_apply_adam (shard_peer.cu,
// each owner sweeps its own shard).  A sweep kernel maps the tile's rows that have a gradient into a shared-memory
// map (s_map[r - r0] >= 0: a key naming where the row's gradient is; -1: none), then runs adam_tile.
#pragma once
#include "common.cuh"
#include "update.cuh"

namespace dir {

constexpr int kAdamTile = 1024;        // table rows per tile (one shared-memory map of distinct-row indices)
constexpr int kAdamThreads = 256;
constexpr int kAdamUnroll = 2;         // float4 chunks each thread loads before it stores any

// first u in [0, n) with a[u] >= key (a ascending), by one warp: 32 probes per round, so ~log32(n) rounds
__device__ __forceinline__ int64_t warp_lower_bound(const uint32_t* __restrict__ a, int64_t n, uint64_t key) {
  const int lane = threadIdx.x & 31;
  int64_t lo = 0, hi = n;   // the answer lies in [lo, hi]
  while (lo < hi) {
    const int64_t step = (hi - lo + 31) / 32;
    const int64_t p = lo + (int64_t)lane * step;
    const bool less = p < hi && (uint64_t)__ldg(a + p) < key;
    const int c = __popc(__ballot_sync(0xffffffffu, less));   // probes below key: a prefix of the lanes
    if (c == 0) break;
    const int64_t nhi = lo + (int64_t)c * step;
    lo = lo + (int64_t)(c - 1) * step + 1;
    hi = nhi < hi ? nhi : hi;
  }
  return lo;
}

struct AdamStep {
  float lr_t, b1, b2, omb1, omb2, eps;  // omb = 1 - beta, in fp32 as TF evaluates it
};

// lr_t = lr * sqrt(1 - beta2_power) / (1 - beta1_power) from the device-resident powers as they stand
__device__ __forceinline__ AdamStep adam_step(float lr, float b1, float b2, float eps, const float* beta_power) {
  AdamStep s;
  const float p1 = beta_power[0], p2 = beta_power[1];
  s.lr_t = __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.f, p2))), __fsub_rn(1.f, p1));
  s.b1 = b1;
  s.b2 = b2;
  s.omb1 = __fsub_rn(1.f, b1);
  s.omb2 = __fsub_rn(1.f, b2);
  s.eps = eps;
  return s;
}

// one component: decay, add the gradient if the row has one, update T.  IEEE sqrt and divide; no contraction.
__device__ __forceinline__ void adam1(float& t, float& m, float& v, float g, bool has_g, const AdamStep& s) {
  m = __fmul_rn(m, s.b1);
  v = __fmul_rn(v, s.b2);
  if (has_g) {
    m = __fadd_rn(m, __fmul_rn(g, s.omb1));
    v = __fadd_rn(v, __fmul_rn(__fmul_rn(g, g), s.omb2));
  }
  t = __fsub_rn(t, __fdiv_rn(__fmul_rn(s.lr_t, m), __fadd_rn(__fsqrt_rn(v), s.eps)));
}

__device__ __forceinline__ bool zero4(const float4& a) { return a.x == 0.f && a.y == 0.f && a.z == 0.f && a.w == 0.f; }

// last field whose offset <= row
__device__ __forceinline__ int field_of(const int64_t* s_off, int F, uint64_t row) {
  int lo = 0, hi = F;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if ((uint64_t)s_off[mid] <= row) lo = mid; else hi = mid;
  }
  return lo;
}

// The tile body: every row of [r0, r1) decayed, its gradient added where s_map has one, T moved; a row whose m and v
// are zero and that has no gradient is not stored (T - 0 / eps == T bit for bit).  Src supplies the gradient:
//   src.load(key, sub, row) -> float4 `sub` of the row's gradient (issued together with the row's T, m, v loads)
//   src.scale(g, row)       the clip_by_norm factor of the row's column, when the sweep clips
template <int LPR, class Src>
__device__ __forceinline__ void adam_tile(float* table, int64_t row_stride, int64_t r0, int64_t r1,
                                          const int32_t* s_map, const AdamStep& s, const Src& src) {
  constexpr int K = LPR * 4;
  const int n_chunks = (int)(r1 - r0) * LPR;
  for (int c0 = threadIdx.x; c0 < n_chunks; c0 += kAdamThreads * kAdamUnroll) {
    float4 T[kAdamUnroll], M[kAdamUnroll], V[kAdamUnroll], G[kAdamUnroll];
    int uu[kAdamUnroll];
#pragma unroll
    for (int j = 0; j < kAdamUnroll; ++j) {
      const int c = c0 + j * kAdamThreads;
      uu[j] = -1;
      if (c < n_chunks) {
        const int r = c / LPR, sub = c % LPR;
        const float* p = table + (r0 + r) * row_stride + sub * 4;
        T[j] = *reinterpret_cast<const float4*>(p);
        M[j] = *reinterpret_cast<const float4*>(p + K);
        V[j] = *reinterpret_cast<const float4*>(p + 2 * K);
        uu[j] = s_map[r];
        if (uu[j] >= 0) G[j] = src.load(uu[j], sub, r0 + r);
      }
    }
#pragma unroll
    for (int j = 0; j < kAdamUnroll; ++j) {
      const int c = c0 + j * kAdamThreads;
      if (c >= n_chunks) continue;
      const bool has_g = uu[j] >= 0;
      if (!has_g && zero4(M[j]) && zero4(V[j])) continue;   // T, m, v stay as they are, bit for bit
      const int r = c / LPR, sub = c % LPR;
      float4 g = has_g ? G[j] : make_float4(0.f, 0.f, 0.f, 0.f);
      if (has_g) src.scale(g, r0 + r);
      adam1(T[j].x, M[j].x, V[j].x, g.x, has_g, s);
      adam1(T[j].y, M[j].y, V[j].y, g.y, has_g, s);
      adam1(T[j].z, M[j].z, V[j].z, g.z, has_g, s);
      adam1(T[j].w, M[j].w, V[j].w, g.w, has_g, s);
      float* p = table + (r0 + r) * row_stride + sub * 4;
      *reinterpret_cast<float4*>(p) = T[j];
      *reinterpret_cast<float4*>(p + K) = M[j];
      *reinterpret_cast<float4*>(p + 2 * K) = V[j];
    }
  }
}

// clip_by_norm of a gradient float4 by its column's denominator (the factors of clip_denominators in shared memory)
__device__ __forceinline__ void clip4(float4& g, float clip, float den) {
  g.x = clip1(g.x, clip, den);
  g.y = clip1(g.y, clip, den);
  g.z = clip1(g.z, clip, den);
  g.w = clip1(g.w, clip, den);
}

// Adam._finish on `st`, after every reader of this step's powers: beta1_power *= beta1, beta2_power *= beta2 (one
// launch; the caller counts it and checks the launch)
void adam_advance_powers(float* beta_power, float b1, float b2, cudaStream_t st);

}  // namespace dir
