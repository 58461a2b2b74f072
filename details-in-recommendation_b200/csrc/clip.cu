// tf.clip_by_norm on the embedding tables' gradient (models/DeepCrossNetwork/DeepCrossNetwork.py:282-289:
// `grads = [None if g is None else tf.clip_by_norm(g, 100.0) for g in grads]` before apply_gradients).
//
// The reference holds ONE variable per column, and [TF] embedding_lookup_sparse de-duplicates ids before the gather,
// so the gradient of column f is an IndexedSlices whose `values` are the per-distinct-row sums G_r of that column and
// clip_by_norm rescales them by clip / max(||values||_2, clip): one factor PER COLUMN, known only once every row sum
// of the column is.  The fused backward applies a row the moment its run is summed, so the clipped backward runs in
// two passes instead (only when a clip norm is set):
//   dir_embed_bwd_reduce_emit_local   per-distinct-row sums -> gu[u] = (G[K], g1)            (embed_bwd.cu)
//   dir_field_sqnorms                 per column: sum of squares of G and of g1, fixed order, fp64
//   dir_rows_apply_clipped            per distinct row: scale by its column's factor, fused Adagrad / SGD update
// The linear weights of a column are a variable of their own (linear_model, deepFM.py:258-263) and get their own factor.
#include "common.cuh"
#include "update.cuh"

namespace dir {

// first distinct row u with urows[u] >= row (urows ascending, as unsigned)
__device__ __forceinline__ int64_t lower_bound_u32(const uint32_t* __restrict__ a, int64_t n, uint64_t row) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((uint64_t)__ldg(a + mid) < row) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// grid (F, kClipSlices): slice s of column f sums the squares of rows lo + s, lo + s + S, ... in a fixed order
template <int LPR>
__global__ void __launch_bounds__(256)
field_sqnorm_kernel(const float* __restrict__ gu, int64_t stride, const uint32_t* __restrict__ urows,
                    const int64_t* __restrict__ count, const int64_t* __restrict__ field_offset, int F,
                    int64_t n_rows, double* __restrict__ part /*[F][kClipSlices][2]*/) {
  constexpr int K = LPR * 4;
  __shared__ double red[2][256];
  __shared__ int64_t s_lo, s_hi;
  const int f = blockIdx.x, sl = blockIdx.y;
  if (threadIdx.x == 0) {
    const int64_t U = *count;
    const uint64_t r0 = (uint64_t)field_offset[f];
    const uint64_t r1 = f + 1 < F ? (uint64_t)field_offset[f + 1] : (uint64_t)n_rows;
    s_lo = lower_bound_u32(urows, U, r0);
    s_hi = lower_bound_u32(urows, U, r1);
  }
  __syncthreads();
  const int sub = threadIdx.x % LPR;
  const int64_t g = threadIdx.x / LPR;           // row group of this thread
  constexpr int GROUPS = 256 / LPR;
  double sq = 0.0, sq1 = 0.0;
  for (int64_t u = s_lo + sl + (int64_t)kClipSlices * g; u < s_hi; u += (int64_t)kClipSlices * GROUPS) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(gu + u * stride) + sub);
    sq += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
    if (sub == 0) {
      const float g1 = __ldg(gu + u * stride + K);
      sq1 += (double)g1 * g1;
    }
  }
  red[0][threadIdx.x] = sq;
  red[1][threadIdx.x] = sq1;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (threadIdx.x < st) {
      red[0][threadIdx.x] += red[0][threadIdx.x + st];
      red[1][threadIdx.x] += red[1][threadIdx.x + st];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    part[((int64_t)f * kClipSlices + sl) * 2] = red[0][0];
    part[((int64_t)f * kClipSlices + sl) * 2 + 1] = red[1][0];
  }
}


template <int LPR>
__global__ void __launch_bounds__(256)
rows_apply_clipped_kernel(float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum,
                          int64_t lin_stride, const LinOpt lo, const float* __restrict__ gu, int64_t stride,
                          const uint32_t* __restrict__ urows, const int64_t* __restrict__ count,
                          const int64_t* __restrict__ field_offset, int F, const double* __restrict__ part,
                          float clip, int opt, float lr, int64_t* n_unique_out) {
  constexpr int K = LPR * 4;
  __shared__ int64_t s_off[kClipMaxFields];
  __shared__ float s_den[kClipMaxFields], s_den1[kClipMaxFields];
  clip_denominators(part, field_offset, F, clip, s_off, s_den, s_den1);
  __syncthreads();
  const int64_t U = *count;
  if (n_unique_out && blockIdx.x == 0 && threadIdx.x == 0) *n_unique_out = U;
  const bool adagrad = opt == DIR_OPT_ADAGRAD;
  const int sub = threadIdx.x % LPR;
  const int64_t step = ((int64_t)gridDim.x * blockDim.x) / LPR;
  for (int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR; u < U; u += step) {
    const uint64_t row = __ldg(urows + u);
    int lo_f = 0, hi_f = F;  // last field whose offset <= row
    while (hi_f - lo_f > 1) {
      const int mid = (lo_f + hi_f) >> 1;
      if ((uint64_t)s_off[mid] <= row) lo_f = mid; else hi_f = mid;
    }
    const float den = s_den[lo_f];
    float4 g = __ldg(reinterpret_cast<const float4*>(gu + u * stride) + sub);
    g.x = clip1(g.x, clip, den);
    g.y = clip1(g.y, clip, den);
    g.z = clip1(g.z, clip, den);
    g.w = clip1(g.w, clip, den);
    const int64_t ro = (int64_t)row * row_stride;
    float4 T = *(reinterpret_cast<const float4*>(table + ro) + sub);
    float4 A = make_float4(0.f, 0.f, 0.f, 0.f);
    if (adagrad) A = *(reinterpret_cast<const float4*>(accum + ro) + sub);
    T.x = upd(T.x, g.x, lr, A.x, adagrad);
    T.y = upd(T.y, g.y, lr, A.y, adagrad);
    T.z = upd(T.z, g.z, lr, A.z, adagrad);
    T.w = upd(T.w, g.w, lr, A.w, adagrad);
    *(reinterpret_cast<float4*>(table + ro) + sub) = T;
    if (adagrad) *(reinterpret_cast<float4*>(accum + ro) + sub) = A;
    if (lin != nullptr && sub == 0) {
      const float g1 = clip1(__ldg(gu + u * stride + K), clip, s_den1[lo_f]);
      const int64_t off = (int64_t)row * lin_stride;
      float n1, z1;
      lin_load(lo, lin_accum, off, n1, z1);
      lin_apply(lo, lin + off, lin_accum + off, lo.z + off, lin[off], n1, z1, g1);
    }
  }
}

}  // namespace dir

extern "C" size_t dir_field_sqnorms_bytes(int F) {
  return F > 0 ? (size_t)F * dir::kClipSlices * 2 * sizeof(double) : 0;
}

extern "C" int dir_field_sqnorms(const float* gu, int64_t gu_stride, const uint32_t* unique_rows,
                                 const int64_t* n_unique_dev, const int64_t* field_offset, int F, int K,
                                 int64_t n_rows, double* partials, dir_stream_t stream) {
  using namespace dir;
  if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "field_sqnorms: 0 < F <= 1024 required");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "field_sqnorms: K must be one of 4, 8, 16, 32, 64");
  if (!gu || !unique_rows || !n_unique_dev || !field_offset || !partials)
    return fail(DIR_EINVAL, "field_sqnorms: null pointer");
  if (gu_stride < K + 1 || (gu_stride & 3) || !aligned16(gu))
    return fail(DIR_EINVAL, "field_sqnorms: gu must be 16-byte aligned, gu_stride >= K + 1 and a multiple of 4");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 grid((unsigned)F, kClipSlices);
#define DIR_SQ(LP) field_sqnorm_kernel<LP><<<grid, 256, 0, st>>>(gu, gu_stride, unique_rows, n_unique_dev, field_offset, F, n_rows, partials)
  switch (K / 4) {
    case 1: DIR_SQ(1); break;
    case 2: DIR_SQ(2); break;
    case 4: DIR_SQ(4); break;
    case 8: DIR_SQ(8); break;
    default: DIR_SQ(16); break;
  }
#undef DIR_SQ
  return launched("field_sqnorms");
}

extern "C" int dir_rows_apply_clipped(float* table, float* accum, int64_t row_stride, float* lin, float* lin_accum,
                                      int64_t lin_stride, const float* gu, int64_t gu_stride,
                                      const uint32_t* unique_rows, const int64_t* n_unique_dev, int64_t n_capacity,
                                      const int64_t* field_offset, int F, int K, const double* partials,
                                      float clip_norm, int optimizer, float lr, const dir_linear_opt* linear_opt,
                                      int64_t* n_unique_out, dir_stream_t stream) {
  using namespace dir;
  if (F <= 0 || F > kClipMaxFields) return fail(DIR_EINVAL, "rows_apply_clipped: 0 < F <= 1024 required");
  if (K != 4 && K != 8 && K != 16 && K != 32 && K != 64)
    return fail(DIR_EINVAL, "rows_apply_clipped: K must be one of 4, 8, 16, 32, 64");
  if (optimizer != DIR_OPT_SGD && optimizer != DIR_OPT_ADAGRAD)
    return fail(DIR_EINVAL, "rows_apply_clipped: unknown optimizer");
  if (!(clip_norm > 0.f)) return fail(DIR_EINVAL, "rows_apply_clipped: clip_norm must be > 0");
  if (!table || !gu || !unique_rows || !n_unique_dev || !field_offset || !partials || n_capacity < 0)
    return fail(DIR_EINVAL, "rows_apply_clipped: null pointer");
  if (optimizer == DIR_OPT_ADAGRAD && !accum) return fail(DIR_EINVAL, "rows_apply_clipped: Adagrad needs accum");
  if (row_stride < K || (row_stride & 3) || gu_stride < K + 1 || (gu_stride & 3))
    return fail(DIR_EINVAL, "rows_apply_clipped: strides must be multiples of 4, >= K (rows), >= K + 1 (gu)");
  if (!aligned16(table) || !aligned16(accum) || !aligned16(gu))
    return fail(DIR_EINVAL, "rows_apply_clipped: table, accum, gu must be 16-byte aligned");
  LinOpt lo;
  if (int rc = resolve_lin("rows_apply_clipped", linear_opt, optimizer, lr, lin, lin_accum, lo)) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t want = (n_capacity * (K / 4) + 255) / 256;
  const unsigned grid = (unsigned)(want < 1 ? 1 : (want < (int64_t)kSMs * 16 ? want : (int64_t)kSMs * 16));
#define DIR_AC(LP)                                                                                              \
  rows_apply_clipped_kernel<LP><<<grid, 256, 0, st>>>(table, accum, row_stride, lin, lin_accum, lin_stride, lo, gu, \
                                                      gu_stride, unique_rows, n_unique_dev, field_offset, F, partials, \
                                                      clip_norm, optimizer, lr, n_unique_out)
  switch (K / 4) {
    case 1: DIR_AC(1); break;
    case 2: DIR_AC(2); break;
    case 4: DIR_AC(4); break;
    case 8: DIR_AC(8); break;
    default: DIR_AC(16); break;
  }
#undef DIR_AC
  return launched("rows_apply_clipped");
}
