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
#include "adam.cuh"

namespace dir {

// Src of adam_tile: the gradient of distinct row uu at gu + uu * gu_stride, clipped by its column's factor
struct UniqueGrad {
  const float* __restrict__ gu;
  int64_t gu_stride;
  bool clipped;
  const int64_t* s_off;
  int F;
  float clip;
  const float* s_den;
  __device__ __forceinline__ float4 load(int uu, int sub, int64_t) const {
    return __ldg(reinterpret_cast<const float4*>(gu + (int64_t)uu * gu_stride) + sub);
  }
  __device__ __forceinline__ void scale(float4& g, int64_t row) const {
    if (clipped) clip4(g, clip, s_den[field_of(s_off, F, (uint64_t)row)]);
  }
};

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
  const AdamStep s = adam_step(lr, b1, b2, eps, beta_power);
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
    adam_tile<LPR>(table, row_stride, r0, r1, s_map, s, UniqueGrad{gu, gu_stride, clipped, s_off, F, clip, s_den});
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

void adam_advance_powers(float* beta_power, float b1, float b2, cudaStream_t st) {
  adam_advance_powers_kernel<<<1, 1, 0, st>>>(beta_power, b1, b2);
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
