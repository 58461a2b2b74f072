// [TF] tf.train.AdamOptimizer on an embedding table's IndexedSlices gradient (the reference's DCN optimizer,
// models/DeepCrossNetwork/train.py:104-124, DeepCrossNetwork.py:264-290).  _apply_sparse_shared runs over the WHOLE
// variable, not just the rows of the batch:
//   lr_t = lr * sqrt(1 - beta2_power) / (1 - beta1_power)        the powers as they stand before this step
//   m = m * beta1;              m[r] += g_r * (1 - beta1)         every row decays; the batch's rows scatter-add
//   v = v * beta2;              v[r] += (g_r * g_r) * (1 - beta2)
//   T = T - (lr_t * m) / (sqrt(v) + epsilon)                      every row (epsilon outside the sqrt)
//   _finish: beta1_power *= beta1, beta2_power *= beta2
// So one apply is a sweep of all n_rows rows [T | m | v]: the kernel walks the table in tiles, finds the slice of the
// ascending distinct-row list that falls in each tile, maps it into shared memory and updates every row of the tile,
// adding the gradient where the row has one.  The clip_by_norm factor of a column comes from dir_field_sqnorms'
// partials exactly as in dir_rows_apply_clipped (clip.cu).  A row whose m and v are zero and that has no gradient
// does not move (T - 0 / eps == T bit for bit), so its stores are skipped.
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

template <int LPR>
__global__ void __launch_bounds__(kAdamThreads, 4)
rows_apply_adam_kernel(float* table, int64_t row_stride, int64_t n_rows, float* lin, float* lin_accum,
                       int64_t lin_stride, const LinOpt lo, const float* __restrict__ gu, int64_t gu_stride,
                       const uint32_t* __restrict__ urows, const int64_t* __restrict__ count, int64_t n_capacity,
                       const int64_t* __restrict__ field_offset, int F, const double* __restrict__ part, float clip,
                       float lr, float b1, float b2, float eps, const float* __restrict__ beta_power,
                       int64_t* n_unique_out) {
  constexpr int K = LPR * 4;
  __shared__ int32_t s_map[kAdamTile];
  __shared__ int64_t s_range[2];
  __shared__ int64_t s_off[kClipMaxFields];
  __shared__ float s_den[kClipMaxFields], s_den1[kClipMaxFields];
  const bool clipped = part != nullptr;
  if (clipped) clip_denominators(part, field_offset, F, clip, s_off, s_den, s_den1);  // published by the first tile's sync
  int64_t U = 0;
  if (n_capacity > 0) {
    U = *count;
    U = U < 0 ? 0 : (U > n_capacity ? n_capacity : U);
  }
  if (n_unique_out && blockIdx.x == 0 && threadIdx.x == 0) *n_unique_out = U;
  AdamStep s;
  {
    const float p1 = beta_power[0], p2 = beta_power[1];
    s.lr_t = __fdiv_rn(__fmul_rn(lr, __fsqrt_rn(__fsub_rn(1.f, p2))), __fsub_rn(1.f, p1));
    s.b1 = b1;
    s.b2 = b2;
    s.omb1 = __fsub_rn(1.f, b1);
    s.omb2 = __fsub_rn(1.f, b2);
    s.eps = eps;
  }
  const int warp = threadIdx.x >> 5;
  const int64_t n_tiles = (n_rows + kAdamTile - 1) / kAdamTile;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * kAdamTile;
    const int64_t r1 = r0 + kAdamTile < n_rows ? r0 + kAdamTile : n_rows;
    if (warp < 2) {                       // warp 0: first distinct row >= r0, warp 1: first >= r1
      const int64_t b = warp_lower_bound(urows, U, (uint64_t)(warp == 0 ? r0 : r1));
      if ((threadIdx.x & 31) == 0) s_range[warp] = b;
    }
    for (int i = threadIdx.x; i < kAdamTile; i += blockDim.x) s_map[i] = -1;
    __syncthreads();                      // also publishes the clip factors on the first tile
    const int64_t ulo = s_range[0], uhi = s_range[1];
    for (int64_t u = ulo + threadIdx.x; u < uhi; u += blockDim.x) s_map[__ldg(urows + u) - r0] = (int32_t)u;
    __syncthreads();
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
          if (uu[j] >= 0) G[j] = __ldg(reinterpret_cast<const float4*>(gu + (int64_t)uu[j] * gu_stride) + sub);
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
        if (has_g && clipped) {
          const float den = s_den[field_of(s_off, F, (uint64_t)(r0 + r))];
          g.x = clip1(g.x, clip, den);
          g.y = clip1(g.y, clip, den);
          g.z = clip1(g.z, clip, den);
          g.w = clip1(g.w, clip, den);
        }
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
    if (lin != nullptr) {                 // first-order weights of the tile's rows that have a gradient
      for (int64_t u = ulo + threadIdx.x; u < uhi; u += blockDim.x) {
        const uint64_t row = __ldg(urows + u);
        float g1 = __ldg(gu + u * gu_stride + K);
        if (clipped) g1 = clip1(g1, clip, s_den1[field_of(s_off, F, row)]);
        const int64_t off = (int64_t)row * lin_stride;
        float n1, z1;
        lin_load(lo, lin_accum, off, n1, z1);
        lin_apply(lo, lin + off, lin_accum + off, lo.z + off, lin[off], n1, z1, g1);
      }
    }
    __syncthreads();                      // s_map / s_range are rewritten by the next tile
  }
}

// _finish: after every reader of this step's powers (same stream)
__global__ void adam_advance_powers_kernel(float* beta_power, float b1, float b2) {
  beta_power[0] = __fmul_rn(beta_power[0], b1);
  beta_power[1] = __fmul_rn(beta_power[1], b2);
}

}  // namespace dir

extern "C" int dir_rows_apply_adam(float* table, int64_t row_stride, int64_t n_rows, int K, float* lin,
                                   float* lin_accum, int64_t lin_stride, const dir_linear_opt* linear_opt,
                                   const float* gu, int64_t gu_stride, const uint32_t* unique_rows,
                                   const int64_t* n_unique_dev, int64_t n_capacity, const int64_t* field_offset, int F,
                                   const double* partials, float clip_norm, const dir_adam_opt* adam,
                                   int64_t* n_unique_out, dir_stream_t stream) {
  using namespace dir;
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "rows_apply_adam: K must be one of 4, 8, 16, 32, 64");
  if (n_rows <= 0 || n_rows >= 0xffffffffLL) return fail(DIR_EINVAL, "rows_apply_adam: 0 < n_rows < 2^32 - 1 required");
  if (!table || !adam || !adam->beta_power) return fail(DIR_EINVAL, "rows_apply_adam: null pointer");
  if (row_stride < 3 * K || (row_stride & 3) || !aligned16(table))
    return fail(DIR_EINVAL, "rows_apply_adam: rows are [T | m | v]: row_stride >= 3K, a multiple of 4, table 16-byte aligned");
  if (!(adam->lr > 0.f)) return fail(DIR_EINVAL, "rows_apply_adam: lr must be > 0");
  if (!(adam->beta1 >= 0.f && adam->beta1 < 1.f) || !(adam->beta2 >= 0.f && adam->beta2 < 1.f))
    return fail(DIR_EINVAL, "rows_apply_adam: 0 <= beta1, beta2 < 1 required");
  if (!(adam->epsilon > 0.f)) return fail(DIR_EINVAL, "rows_apply_adam: epsilon must be > 0");
  if (n_capacity < 0) return fail(DIR_EINVAL, "rows_apply_adam: n_capacity must be >= 0");
  if (n_capacity > 0) {
    if (!gu || !unique_rows || !n_unique_dev) return fail(DIR_EINVAL, "rows_apply_adam: null pointer");
    if (gu_stride < K + 1 || (gu_stride & 3) || !aligned16(gu))
      return fail(DIR_EINVAL, "rows_apply_adam: gu must be 16-byte aligned, gu_stride >= K + 1 and a multiple of 4");
  }
  if (partials) {
    if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "rows_apply_adam: 0 < F <= 1024 required");
    if (!field_offset) return fail(DIR_EINVAL, "rows_apply_adam: the clip needs field_offset");
    if (!(clip_norm > 0.f)) return fail(DIR_EINVAL, "rows_apply_adam: clip_norm must be > 0");
  }
  LinOpt lo{DIR_OPT_SGD, 0.f, 0.f, 0.f, nullptr};
  if (lin != nullptr) {
    if (!linear_opt) return fail(DIR_EINVAL, "rows_apply_adam: lin needs linear_opt (Adam does not train first-order weights)");
    if (int rc = resolve_lin("rows_apply_adam", linear_opt, DIR_OPT_SGD, 0.f, lin, lin_accum, lo)) return rc;
    if (lin_stride < 1) return fail(DIR_EINVAL, "rows_apply_adam: lin_stride must be >= 1");
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n_tiles = (n_rows + kAdamTile - 1) / kAdamTile;
  const unsigned grid = (unsigned)(n_tiles < (int64_t)kSMs * 4 ? n_tiles : (int64_t)kSMs * 4);
  const float b1 = adam->beta1, b2 = adam->beta2;
#define DIR_AD(LP)                                                                                                   \
  rows_apply_adam_kernel<LP><<<grid, kAdamThreads, 0, st>>>(table, row_stride, n_rows, lin, lin_accum, lin_stride, lo, \
                                                            gu, gu_stride, unique_rows, n_unique_dev, n_capacity,     \
                                                            field_offset, F, partials, clip_norm, adam->lr, b1, b2,   \
                                                            adam->epsilon, adam->beta_power, n_unique_out)
  switch (K / 4) {
    case 1: DIR_AD(1); break;
    case 2: DIR_AD(2); break;
    case 4: DIR_AD(4); break;
    case 8: DIR_AD(8); break;
    default: DIR_AD(16); break;
  }
#undef DIR_AD
  adam_advance_powers_kernel<<<1, 1, 0, st>>>(adam->beta_power, b1, b2);
  return launched("rows_apply_adam", 2);
}
