// K4+K5: DCN-v1 cross stack  x_{l+1} = (x0 * (x_l . w_l) + b_l) + x_l,  all L layers in one pass.
// Not a GEMM (the per-layer "matvec" is one dot product per sample), so no tensor cores: the kernels
// are HBM-bound streams over x0 / dy with the per-sample work done by one warp in registers.
//
// Both directions use the rank-1 structure of the recurrence.  With  p_l = x0 . w_l  (per sample),
// beta_l = sum_{j<l} b_j  (per column) and  q_l = beta_l . w_l  (one scalar per layer):
//     x_l = x0 * c_l + beta_l,      s_l = x_l . w_l = c_l p_l + q_l,      c_{l+1} = c_l + s_l,  c_0 = 1
// so the forward is L dot products of x0 with the w_l, a scalar recurrence, and one fused
// multiply-add per output element ( x_L = x0 * c_L + beta_L ): 7 FMAs per element at L = 6 instead of
// the 18 flops + 12 parameter loads of the layer-by-layer sweep, which was issue-bound (ncu: 0.64 IPC
// per scheduler, 31 % DRAM; profiles/r01_kernels_v3_ncu.txt).  The backward, with a = dy . x0 :
//     ds_l = a + sum_{j>l} ds_j p_j                       (scalar recurrence, l = L-1 .. 0)
//     dx0  = c_L dy + sum_l (ds_l c_l) w_l
//     dw_l = sum_b (ds_l c_l) x0  +  beta_l * sum_b ds_l
//     db_l = sum_b dy  +  sum_{j>l} w_j * sum_b ds_j
// No x_l is ever stored.  Batch sums are reduced in a fixed order (per-thread sequential over the
// CTA's tiles, per-CTA partials combined by one finishing kernel): deterministic, no float atomics.
// Results differ from the reference's ((x0*s)+b)+x evaluation order by rounding only (a few ulp of
// the largest term; the parity tests hold 1e-5 relative against the fp64 oracle).
//
// Reference: models/DeepCrossNetwork/DeepCrossNetwork.py:336-367 and TF autodiff of it (:283).
#include <algorithm>

#include "common.cuh"

namespace dir {

template <int VEC>
struct Pack {
  float v[VEC];
};
template <int VEC>
__device__ __forceinline__ Pack<VEC> ld_pack(const float* p, bool stream) {
  Pack<VEC> r;
  if constexpr (VEC == 4) {
    const float4 t = stream ? ldg_stream(p) : __ldg(reinterpret_cast<const float4*>(p));
    r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
  } else {
    r.v[0] = __ldg(p);
  }
  return r;
}
template <int VEC>
__device__ __forceinline__ void st_pack(float* p, const float* v) {
  if constexpr (VEC == 4) {
    stg_stream(p, make_float4(v[0], v[1], v[2], v[3]));
  } else {
    *p = v[0];
  }
}

constexpr int kCrossWarps = 8;  // warps per CTA

// ------------------------------------------------------------------------------ per-CTA constants
// beta_L[c] = sum_l b_l[c] (layer order) and q_l = beta_l . w_l, computed once per CTA by its 256
// threads in a fixed order (thread t owns columns t, t+256, ...; warp sums, then warps in order).
// s_beta may be NULL.  Ends with a __syncthreads().
__device__ __forceinline__ void cross_constants(const float* __restrict__ wg,
                                                const float* __restrict__ bg, int d, int L,
                                                float* s_beta, float* s_q, float* s_red) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  float beta[4] = {0.f, 0.f, 0.f, 0.f};  // d <= 1024 = 4 * 256
  for (int l = 0; l < L; ++l) {
    float part = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = threadIdx.x + j * 256;
      if (c < d) {
        part = fmaf(beta[j], __ldg(wg + l * d + c), part);
        beta[j] += __ldg(bg + l * d + c);
      }
    }
    part = warp_sum(part);
    if (lane == 0) s_red[wib] = part;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < kCrossWarps; ++w) t += s_red[w];
      s_q[l] = t;
    }
    __syncthreads();
  }
  if (s_beta != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = threadIdx.x + j * 256;
      if (c < d) s_beta[c] = beta[j];
    }
  }
  __syncthreads();
}

// w[L][d] -> shared memory as [L][DP], DP = 32 lanes * E columns, zero beyond d: the per-layer loads
// become unpredicated LDS.128 at lane * 16 + constant offsets (the global loads cost ~7 issue slots each
// in address arithmetic, predicates and selects: profiles/r01_cross_v4_ncu.txt).  Caller syncs.
template <int DP>
__device__ __forceinline__ void stage_w(const float* __restrict__ wg, int d, int L, float* s_w) {
  for (int t = threadIdx.x; t < L * DP; t += blockDim.x) {
    const int l = t / DP, c = t - l * DP;
    s_w[t] = c < d ? __ldg(wg + l * d + c) : 0.f;
  }
}
template <int VEC>
__device__ __forceinline__ Pack<VEC> lds_pack(const float* p) {
  Pack<VEC> r;
  if constexpr (VEC == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    r.v[0] = t.x; r.v[1] = t.y; r.v[2] = t.z; r.v[3] = t.w;
  } else {
    r.v[0] = *p;
  }
  return r;
}

// ------------------------------------------------------------------------------ forward
// One warp per PAIR of samples (the w_l loads are shared by the pair), persistent grid.
// pg [B,L] (nullable) receives p_l = x0 . w_l for the backward.
template <int VEC, int NPL, bool WSMEM>
__global__ void __launch_bounds__(kCrossWarps * 32)
cross_fwd_kernel(const float* __restrict__ x0g, const float* __restrict__ wg,
                 const float* __restrict__ bg, int64_t B, int d, int L, float* __restrict__ xLg,
                 float* __restrict__ pg) {
  constexpr int E = VEC * NPL;
  constexpr int DP = E * 32;
  __shared__ float s_beta[1024];
  __shared__ float s_q[32];
  __shared__ float s_red[kCrossWarps];
  extern __shared__ __align__(16) float s_w[];  // [L][DP] when WSMEM
  if (WSMEM) stage_w<DP>(wg, d, L, s_w);
  cross_constants(wg, bg, d, L, s_beta, s_q, s_red);
  const int lane = threadIdx.x & 31;
  const float q_mine = lane < L ? s_q[lane] : 0.f;
  float betaL[E];
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int c = (i * 32 + lane) * VEC;
#pragma unroll
    for (int e = 0; e < VEC; ++e) betaL[i * VEC + e] = (c + e < d) ? s_beta[c + e] : 0.f;
  }
  const int64_t pair0 = (int64_t)blockIdx.x * kCrossWarps + (threadIdx.x >> 5);
  const int64_t npairs = (int64_t)gridDim.x * kCrossWarps;
  for (int64_t b = pair0 * 2; b < B; b += npairs * 2) {
    const bool two = b + 1 < B;
    float xa[E], xb[E];
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      Pack<VEC> pa{}, pb{};
      if (c < d) {
        pa = ld_pack<VEC>(x0g + b * d + c, true);
        if (two) pb = ld_pack<VEC>(x0g + (b + 1) * d + c, true);
      }
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        xa[i * VEC + e] = (c < d) ? pa.v[e] : 0.f;
        xb[i * VEC + e] = (c < d && two) ? pb.v[e] : 0.f;
      }
    }
    float ca = 1.f, cb = 1.f;  // c_l = 1 + sum_{j<l} s_j
    for (int l = 0; l < L; ++l) {
      float da = 0.f, db = 0.f;
      const float* wl = s_w + l * DP + lane * VEC;
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = (i * 32 + lane) * VEC;
        Pack<VEC> pw{};
        if (WSMEM) {
          pw = lds_pack<VEC>(wl + i * 32 * VEC);
        } else if (c < d) {
          pw = ld_pack<VEC>(wg + l * d + c, false);
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const float wv = (WSMEM || c < d) ? pw.v[e] : 0.f;
          da = fmaf(xa[i * VEC + e], wv, da);
          db = fmaf(xb[i * VEC + e], wv, db);
        }
      }
      da = warp_sum(da);
      db = warp_sum(db);
      const float q = __shfl_sync(0xffffffffu, q_mine, l);
      if (pg && lane == 0) {
        pg[b * L + l] = da;
        if (two) pg[(b + 1) * L + l] = db;
      }
      ca += fmaf(ca, da, q);  // s_l = c_l p_l + q_l
      cb += fmaf(cb, db, q);
    }
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      float oa[VEC], ob[VEC];
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        oa[e] = fmaf(xa[i * VEC + e], ca, betaL[i * VEC + e]);  // x_L = x0 c_L + beta_L
        ob[e] = fmaf(xb[i * VEC + e], cb, betaL[i * VEC + e]);
      }
      if (c < d) {
        st_pack<VEC>(xLg + b * d + c, oa);
        if (two) st_pack<VEC>(xLg + (b + 1) * d + c, ob);
      }
    }
  }
}

// ------------------------------------------------------------------------------ backward
struct CrossBwdWs {
  float* alpha;   // [B][L]   ds_l * c_l
  float* Dpart;   // [G1][L]  per-CTA sum_b ds_l
  float* dypart;  // [G1][d]  per-CTA sum_b dy
  float* dwpart;  // [G2][L][d] per-CTA sum_b alpha_l x0
  int G1, G2;
  size_t total;
};

static int cross_grid1(int64_t B) {
  const int64_t want = (B + kCrossWarps - 1) / kCrossWarps;
  const int64_t cap = kSMs * 4;
  return (int)(want < cap ? want : cap);
}
static int cross_grid_fused(int64_t B) {  // persistent: two CTAs per SM
  const int64_t want = (B + 15) / 16;
  const int64_t cap = kSMs * 2;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}
static int cross_grid2(int64_t B) {
  const int64_t want = (B + 31) / 32;
  const int64_t cap = kSMs * 4;
  return (int)(want < cap ? (want > 0 ? want : 1) : cap);
}

static CrossBwdWs cross_carve(void* base, int64_t B, int d, int L) {
  CrossBwdWs w;
  char* p = static_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    char* r = p ? p + off : nullptr;
    off += align_up(bytes, 256);
    return reinterpret_cast<float*>(r);
  };
  const bool fused = L <= 8;
  w.G1 = fused ? cross_grid_fused(B) : cross_grid1(B);
  w.G2 = fused ? w.G1 : cross_grid2(B);
  w.alpha = take(fused ? 0 : (size_t)B * L * 4);
  w.Dpart = take((size_t)w.G1 * L * 4);
  w.dypart = take((size_t)w.G1 * d * 4);
  w.dwpart = take((size_t)w.G2 * L * d * 4);
  w.total = off;
  return w;
}

// pass 1: per-sample sweep -> dx0, alpha, and per-CTA partials of sum ds_l and sum dy
template <int VEC, int NPL>
__global__ void __launch_bounds__(kCrossWarps * 32)
cross_bwd_sample_kernel(const float* __restrict__ x0g, const float* __restrict__ wg,
                        const float* __restrict__ bg, const float* __restrict__ dyg,
                        const float* __restrict__ sg, int64_t B, int d, int L,
                        float* __restrict__ dx0g, float* __restrict__ alpha,
                        float* __restrict__ Dpart, float* __restrict__ dypart) {
  constexpr int E = VEC * NPL;
  extern __shared__ float smem[];  // [kCrossWarps][d] then [kCrossWarps][32]
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int64_t warp0 = (int64_t)blockIdx.x * kCrossWarps + wib;
  const int64_t nwarps = (int64_t)gridDim.x * kCrossWarps;
  float accDy[E];
#pragma unroll
  for (int e = 0; e < E; ++e) accDy[e] = 0.f;
  float Dacc = 0.f;  // lane l: sum over this warp's samples of ds_l

  for (int64_t b = warp0; b < B; b += nwarps) {
    float x0[E], dx[E], dx0[E];
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      Pack<VEC> px{}, pd{};
      if (c < d) {
        px = ld_pack<VEC>(x0g + b * d + c, true);
        pd = ld_pack<VEC>(dyg + b * d + c, true);
      }
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        x0[i * VEC + e] = (c < d) ? px.v[e] : 0.f;
        dx[i * VEC + e] = (c < d) ? pd.v[e] : 0.f;
        dx0[i * VEC + e] = 0.f;
        accDy[i * VEC + e] += dx[i * VEC + e];
      }
    }
    // s_l = x_l . w_l : lane l keeps s_l.  Saved by the forward, or recomputed here.
    float s_mine = 0.f;
    if (sg) {
      if (lane < L) s_mine = __ldg(sg + b * L + lane);
    } else {
      float xl[E];
#pragma unroll
      for (int e = 0; e < E; ++e) xl[e] = x0[e];
      for (int l = 0; l < L; ++l) {
        float dot = 0.f;
        float bv[E];
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const int c = (i * 32 + lane) * VEC;
          Pack<VEC> pw{}, pb{};
          if (c < d) {
            pw = ld_pack<VEC>(wg + l * d + c, false);
            pb = ld_pack<VEC>(bg + l * d + c, false);
          }
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            dot = fmaf(xl[i * VEC + e], (c < d) ? pw.v[e] : 0.f, dot);
            bv[i * VEC + e] = (c < d) ? pb.v[e] : 0.f;
          }
        }
        dot = warp_sum(dot);
#pragma unroll
        for (int e = 0; e < E; ++e)
          xl[e] = __fadd_rn(__fadd_rn(__fmul_rn(x0[e], dot), bv[e]), xl[e]);
        if (lane == l) s_mine = dot;
      }
    }
    // c_l = 1 + sum_{j<l} s_j  (lane l keeps c_l)
    float c_mine = 1.f;
    for (int j = 0; j < L; ++j) {
      const float sj = __shfl_sync(0xffffffffu, s_mine, j);
      if (lane > j) c_mine += sj;
    }
    float alpha_mine = 0.f;
    for (int l = L - 1; l >= 0; --l) {
      const float s_l = __shfl_sync(0xffffffffu, s_mine, l);
      const float c_l = __shfl_sync(0xffffffffu, c_mine, l);
      float ds = 0.f;
#pragma unroll
      for (int e = 0; e < E; ++e) ds = fmaf(dx[e], x0[e], ds);
      ds = warp_sum(ds);
      if (lane == l) {
        alpha_mine = ds * c_l;
        Dacc += ds;
      }
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = (i * 32 + lane) * VEC;
        Pack<VEC> pw{};
        if (c < d) pw = ld_pack<VEC>(wg + l * d + c, false);
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          dx0[i * VEC + e] = fmaf(dx[i * VEC + e], s_l, dx0[i * VEC + e]);
          dx[i * VEC + e] = fmaf(ds, (c < d) ? pw.v[e] : 0.f, dx[i * VEC + e]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      float o[VEC];
#pragma unroll
      for (int e = 0; e < VEC; ++e) o[e] = dx0[i * VEC + e] + dx[i * VEC + e];
      if (c < d) st_pack<VEC>(dx0g + b * d + c, o);
    }
    if (lane < L) alpha[b * L + lane] = alpha_mine;
  }

  // per-CTA partials, warps added in warp order
  float* sdy = smem;
  float* sD = smem + kCrossWarps * d;
#pragma unroll
  for (int i = 0; i < NPL; ++i) {
    const int c = (i * 32 + lane) * VEC;
#pragma unroll
    for (int e = 0; e < VEC; ++e)
      if (c + e < d) sdy[wib * d + c + e] = accDy[i * VEC + e];
  }
  sD[wib * 32 + lane] = Dacc;
  __syncthreads();
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kCrossWarps; ++w) t += sdy[w * d + c];
    dypart[(int64_t)blockIdx.x * d + c] = t;
  }
  if (threadIdx.x < L) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kCrossWarps; ++w) t += sD[w * 32 + threadIdx.x];
    Dpart[(int64_t)blockIdx.x * L + threadIdx.x] = t;
  }
}

// pass 2: dwpart[cta][l][c] = sum over the CTA's samples of alpha[b][l] * x0[b][c]
// thread = one column; samples in sample order.
constexpr int kDwUnroll = 8;
__global__ void __launch_bounds__(256)
cross_bwd_dw_kernel(const float* __restrict__ x0g, const float* __restrict__ alpha, int64_t B,
                    int d, int L, float* __restrict__ dwpart) {
  extern __shared__ float sal[];  // alpha of the current sample block [kDwUnroll][L]
  const int64_t per = (B + gridDim.x - 1) / gridDim.x;
  const int64_t b0 = (int64_t)blockIdx.x * per;
  const int64_t b1 = min(B, b0 + per);
  for (int c0 = 0; c0 < d; c0 += blockDim.x) {
    const int c = c0 + threadIdx.x;
    float acc[8];  // L <= 8 per sweep
    for (int l0 = 0; l0 < L; l0 += 8) {
#pragma unroll
      for (int l = 0; l < 8; ++l) acc[l] = 0.f;
      for (int64_t bb = b0; bb < b1; bb += kDwUnroll) {
        __syncthreads();
        for (int t = threadIdx.x; t < kDwUnroll * 8; t += blockDim.x) {
          const int64_t b = bb + t / 8;
          const int l = l0 + (t & 7);
          sal[t] = (b < b1 && l < L) ? __ldg(alpha + b * L + l) : 0.f;
        }
        __syncthreads();
        float xv[kDwUnroll];
#pragma unroll
        for (int j = 0; j < kDwUnroll; ++j)
          xv[j] = (c < d && bb + j < b1) ? __ldg(x0g + (bb + j) * d + c) : 0.f;
#pragma unroll
        for (int j = 0; j < kDwUnroll; ++j)
#pragma unroll
          for (int l = 0; l < 8; ++l) acc[l] = fmaf(sal[j * 8 + l], xv[j], acc[l]);
      }
      if (c < d)
#pragma unroll
        for (int l = 0; l < 8; ++l)
          if (l0 + l < L) dwpart[((int64_t)blockIdx.x * L + l0 + l) * d + c] = acc[l];
    }
  }
}

// ------------------------------------------------------------------------------ fused backward (L <= 8)
// One pass over x0 and dy.  A CTA walks tiles of kTS samples:
//   phase A  one warp per sample: a = dy . x0, p_l (saved by the forward, or recomputed), the two
//            scalar recurrences (every lane runs them redundantly), dx0 = c_L dy + sum_l alpha_l w_l
//            to HBM, alpha_l = ds_l c_l to shared memory; the warp also leaves its x0 / dy rows in
//            shared memory
//   phase B  one thread per column: dw_l[c] += alpha_l[b] x0[b][c], db[c] += dy[b][c] over the tile,
//            samples in order, accumulators in registers for the whole kernel
// so x0 and dy are read from HBM once.  Per-CTA partials are combined by cross_bwd_finish2_kernel
// in a fixed order.
constexpr int kTS = 16;  // samples per tile: two per warp

template <int VEC, int NPL>
__global__ void __launch_bounds__(kCrossWarps * 32, 2)
cross_bwd_fused_kernel(const float* __restrict__ x0g, const float* __restrict__ wg,
                       const float* __restrict__ bg, const float* __restrict__ dyg,
                       const float* __restrict__ pg, int64_t B, int d, int L,
                       float* __restrict__ dx0g, float* __restrict__ Dpart,
                       float* __restrict__ dypart, float* __restrict__ dwpart) {
  constexpr int E = VEC * NPL;
  constexpr int CI = (E * 32 + 255) / 256;  // columns per thread in phase B
  extern __shared__ float smem[];
  float* x0s = smem;                   // [kTS][d]
  float* dys = x0s + kTS * d;          // [kTS][d]
  float* als = dys + kTS * d;          // [kTS][8]
  float* sD = als + kTS * 8;           // [kCrossWarps][32]
  float* s_q = sD + kCrossWarps * 32;  // [32]
  float* s_red = s_q + 32;             // [kCrossWarps]
  float* s_w = s_red + kCrossWarps;    // [L][DP] zero-padded copy of w
  constexpr int DP = E * 32;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  stage_w<DP>(wg, d, L, s_w);
  cross_constants(wg, bg, d, L, nullptr, s_q, s_red);
  const float q_mine = lane < L ? s_q[lane] : 0.f;
  float acc[CI][8], accdy[CI];
#pragma unroll
  for (int ci = 0; ci < CI; ++ci) {
    accdy[ci] = 0.f;
#pragma unroll
    for (int l = 0; l < 8; ++l) acc[ci][l] = 0.f;
  }
  float Dacc = 0.f;  // lane l: sum over this warp's samples of ds_l

  const int64_t ntiles = (B + kTS - 1) / kTS;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t b0 = tile * kTS;
    // ---- phase A
#pragma unroll 1
    for (int h = 0; h < kTS / kCrossWarps; ++h) {
      const int tb = h * kCrossWarps + wib;
      const int64_t b = b0 + tb;
      float x0[E], dx[E];
      const bool live = b < B;
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        const int c = (i * 32 + lane) * VEC;
        Pack<VEC> px{}, pd{};
        if (live && c < d) {
          px = ld_pack<VEC>(x0g + b * d + c, true);
          pd = ld_pack<VEC>(dyg + b * d + c, true);
        }
#pragma unroll
        for (int e = 0; e < VEC; ++e) {
          const bool in = live && c < d;
          x0[i * VEC + e] = in ? px.v[e] : 0.f;
          dx[i * VEC + e] = in ? pd.v[e] : 0.f;
          a = fmaf(dx[i * VEC + e], x0[i * VEC + e], a);
        }
        if (c < d) {  // the tile copy phase B reads (zeros for samples past the end)
          if constexpr (VEC == 4) {
            *reinterpret_cast<float4*>(x0s + tb * d + c) =
                make_float4(x0[i * 4], x0[i * 4 + 1], x0[i * 4 + 2], x0[i * 4 + 3]);
            *reinterpret_cast<float4*>(dys + tb * d + c) =
                make_float4(dx[i * 4], dx[i * 4 + 1], dx[i * 4 + 2], dx[i * 4 + 3]);
          } else {
            x0s[tb * d + c] = x0[i];
            dys[tb * d + c] = dx[i];
          }
        }
      }
      a = warp_sum(a);
      float p_mine = 0.f;  // lane l keeps p_l = x0 . w_l (0 for l >= L and for samples past the end)
      if (pg) {
        if (live && lane < L) p_mine = __ldg(pg + b * L + lane);
      } else {
        for (int l = 0; l < L; ++l) {
          float dot = 0.f;
          const float* wl = s_w + l * DP + lane * VEC;
#pragma unroll
          for (int i = 0; i < NPL; ++i) {
            const Pack<VEC> pw = lds_pack<VEC>(wl + i * 32 * VEC);
#pragma unroll
            for (int e = 0; e < VEC; ++e) dot = fmaf(x0[i * VEC + e], pw.v[e], dot);
          }
          dot = warp_sum(dot);
          if (lane == l) p_mine = dot;
        }
      }
      // scalar recurrences, every lane redundantly.  Layers l >= L have p = q = 0: c stays, ds = 0.
      float pv[8], cv[9];
      cv[0] = 1.f;
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        pv[l] = __shfl_sync(0xffffffffu, p_mine, l);
        const float q = __shfl_sync(0xffffffffu, q_mine, l);
        cv[l + 1] = cv[l] + fmaf(cv[l], pv[l], q);  // c_{l+1} = c_l + s_l,  s_l = c_l p_l + q_l
      }
      float al[8];  // alpha_l = ds_l c_l
      float t = 0.f, ds_mine = 0.f, al_mine = 0.f;
#pragma unroll
      for (int l = 7; l >= 0; --l) {
        float ds = 0.f;
        if (l < L) {
          ds = a + t;  // ds_l = a + sum_{j>l} ds_j p_j
          t = fmaf(ds, pv[l], t);
        }
        al[l] = ds * cv[l];
        if (lane == l) {
          ds_mine = ds;
          al_mine = al[l];
        }
      }
      Dacc += ds_mine;
      if (lane < 8) als[tb * 8 + lane] = al_mine;
      // dx0 = c_L dy + sum_l alpha_l w_l
      const float cL = cv[8];
#pragma unroll
      for (int e = 0; e < E; ++e) dx[e] *= cL;
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        if (l < L) {  // warp-uniform
          const float* wl = s_w + l * DP + lane * VEC;
#pragma unroll
          for (int i = 0; i < NPL; ++i) {
            const Pack<VEC> pw = lds_pack<VEC>(wl + i * 32 * VEC);
#pragma unroll
            for (int e = 0; e < VEC; ++e) dx[i * VEC + e] = fmaf(al[l], pw.v[e], dx[i * VEC + e]);
          }
        }
      }
      if (live) {
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const int c = (i * 32 + lane) * VEC;
          if (c < d) st_pack<VEC>(dx0g + b * d + c, &dx[i * VEC]);
        }
      }
    }
    __syncthreads();
    // ---- phase B: thread = column, samples of the tile in order
#pragma unroll 4
    for (int tb = 0; tb < kTS; ++tb) {
      const float4 a0 = *reinterpret_cast<const float4*>(als + tb * 8);  // one broadcast load per sample
      const float4 a1 = *reinterpret_cast<const float4*>(als + tb * 8 + 4);
#pragma unroll
      for (int ci = 0; ci < CI; ++ci) {
        const int c = ci * 256 + threadIdx.x;
        if (c < d) {
          const float xv = x0s[tb * d + c];
          acc[ci][0] = fmaf(a0.x, xv, acc[ci][0]);
          acc[ci][1] = fmaf(a0.y, xv, acc[ci][1]);
          acc[ci][2] = fmaf(a0.z, xv, acc[ci][2]);
          acc[ci][3] = fmaf(a0.w, xv, acc[ci][3]);
          acc[ci][4] = fmaf(a1.x, xv, acc[ci][4]);
          acc[ci][5] = fmaf(a1.y, xv, acc[ci][5]);
          acc[ci][6] = fmaf(a1.z, xv, acc[ci][6]);
          acc[ci][7] = fmaf(a1.w, xv, acc[ci][7]);
          accdy[ci] += dys[tb * d + c];
        }
      }
    }
    __syncthreads();
  }
  // per-CTA partials
#pragma unroll
  for (int ci = 0; ci < CI; ++ci) {
    const int c = ci * 256 + threadIdx.x;
    if (c < d) {
      dypart[(int64_t)blockIdx.x * d + c] = accdy[ci];
#pragma unroll
      for (int l = 0; l < 8; ++l)
        if (l < L) dwpart[((int64_t)blockIdx.x * L + l) * d + c] = acc[ci][l];
    }
  }
  sD[wib * 32 + lane] = Dacc;
  __syncthreads();
  if (threadIdx.x < L) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < kCrossWarps; ++w) t += sD[w * 32 + threadIdx.x];
    Dpart[(int64_t)blockIdx.x * L + threadIdx.x] = t;
  }
}

// ------------------------------------------------------------------------------ bulk-copy helpers (1-D TMA)
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------ backward, per-warp rings
// The fastest form, for shapes whose batch sums fit in registers (4 * NPL * (LT + 3) <= 184 floats per lane).
// A warp owns samples gw, gw + W, gw + 2W, ... (W = warps in the grid) and a private ring of `depth` slots in shared
// memory, each holding one x0 row and one dy row.  Lane 0 refills a slot with two bulk asynchronous copies
// (cp.async.bulk, completion counted on the slot's mbarrier) as soon as the warp has moved the slot's rows into
// registers, so depth - 1 rows per warp stay in flight whatever the warp is computing: HBM never waits for a
// phase change, and no __syncthreads() is executed between the prologue and the final combine.  Everything the two
// phases of cross_bwd_fused_kernel did per tile happens on the one register copy of the rows:
//     a, the recurrences, dx0 -> HBM,   acc[l][e] += alpha_l x0[e],   accdy[e] += dy[e]
// i.e. dw / db are accumulated per warp over its own samples in sample order, then the CTA's eight warps are added
// in warp order and the per-CTA partials go to cross_bwd_finish2_kernel as before: fixed order, no float atomics.
// p_l comes from the forward (pg, prefetched one sample ahead) or is recomputed.
constexpr int kRingMaxDepth = 4;

template <int NPL, int LT>
__global__ void __launch_bounds__(kCrossWarps * 32, 1)
cross_bwd_ring_kernel(const float* __restrict__ x0g, const float* __restrict__ wg,
                      const float* __restrict__ bg, const float* __restrict__ dyg,
                      const float* __restrict__ pg, int64_t B, int d, int L, int depth,
                      float* __restrict__ dx0g, float* __restrict__ Dpart,
                      float* __restrict__ dypart, float* __restrict__ dwpart) {
  constexpr int VEC = 4;
  constexpr int E = VEC * NPL;
  constexpr int DP = E * 32;
  extern __shared__ __align__(128) float smem[];
  float* ring = smem;  // [kCrossWarps][depth][x0 row | dy row]; at the end [kCrossWarps][DP] for the combine
  const size_t ring_f = max((size_t)kCrossWarps * depth * 2 * d, (size_t)kCrossWarps * DP);
  float* s_w = ring + ring_f;                               // [L][DP]
  float* sD = s_w + L * DP;                                 // [kCrossWarps][32]
  float* s_q = sD + kCrossWarps * 32;                       // [32]
  float* s_red = s_q + 32;                                  // [kCrossWarps]
  __shared__ __align__(8) uint64_t full[kCrossWarps * kRingMaxDepth];
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const int64_t W = (int64_t)gridDim.x * kCrossWarps;
  const int64_t gw = (int64_t)blockIdx.x * kCrossWarps + wib;
  const int64_t nmine = gw < B ? (B - gw + W - 1) / W : 0;
  const uint32_t row_bytes = (uint32_t)d * 4u;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kCrossWarps * kRingMaxDepth; ++i) mbar_init(&full[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  float* myring = ring + (size_t)wib * depth * 2 * d;
  uint64_t* mybar = full + wib * kRingMaxDepth;
  auto issue = [&](int64_t k, int slot) {  // lane 0 only
    const int64_t b = gw + k * W;
    float* dst = myring + (size_t)slot * 2 * d;
    mbar_expect_tx(&mybar[slot], 2u * row_bytes);
    bulk_g2s(dst, x0g + b * d, row_bytes, &mybar[slot]);
    bulk_g2s(dst + d, dyg + b * d, row_bytes, &mybar[slot]);
  };
  if (lane == 0)
    for (int k = 0; k < depth && k < nmine; ++k) issue(k, k);

  stage_w<DP>(wg, d, L, s_w);
  cross_constants(wg, bg, d, L, nullptr, s_q, s_red);  // ends with a __syncthreads()
  const float q_mine = lane < L ? s_q[lane] : 0.f;
  float acc[LT][E], accdy[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    accdy[e] = 0.f;
#pragma unroll
    for (int l = 0; l < LT; ++l) acc[l][e] = 0.f;
  }
  float Dacc = 0.f;  // lane l: sum over this warp's samples of ds_l
  float p_next = 0.f;
  if (pg && nmine > 0 && lane < L) p_next = __ldg(pg + gw * L + lane);

  int slot = 0;
  uint32_t parity = 0;
#pragma unroll 1
  for (int64_t k = 0; k < nmine; ++k) {
    const int64_t b = gw + k * W;
    mbar_wait(&mybar[slot], parity);
    const float* xs = myring + (size_t)slot * 2 * d;
    float x0[E], dx[E];
    float a = 0.f;
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      float4 px = make_float4(0.f, 0.f, 0.f, 0.f), pd = px;
      if (c < d) {
        px = *reinterpret_cast<const float4*>(xs + c);
        pd = *reinterpret_cast<const float4*>(xs + d + c);
      }
      x0[i * 4] = px.x; x0[i * 4 + 1] = px.y; x0[i * 4 + 2] = px.z; x0[i * 4 + 3] = px.w;
      dx[i * 4] = pd.x; dx[i * 4 + 1] = pd.y; dx[i * 4 + 2] = pd.z; dx[i * 4 + 3] = pd.w;
#pragma unroll
      for (int e = 0; e < VEC; ++e) {
        a = fmaf(dx[i * VEC + e], x0[i * VEC + e], a);
        accdy[i * VEC + e] += dx[i * VEC + e];
      }
    }
    // the rows are in registers: hand the slot back to the copy engine
    __syncwarp();
    if (lane == 0 && k + depth < nmine) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      issue(k + depth, slot);
    }
    if (++slot == depth) {
      slot = 0;
      parity ^= 1u;
    }
    a = warp_sum(a);
    float p_mine = 0.f;  // lane l keeps p_l = x0 . w_l
    if (pg) {
      p_mine = p_next;
      if (k + 1 < nmine && lane < L) p_next = __ldg(pg + (b + W) * L + lane);
    } else {
      for (int l = 0; l < L; ++l) {
        float dot = 0.f;
        const float* wl = s_w + l * DP + lane * VEC;
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const Pack<VEC> pw = lds_pack<VEC>(wl + i * 32 * VEC);
#pragma unroll
          for (int e = 0; e < VEC; ++e) dot = fmaf(x0[i * VEC + e], pw.v[e], dot);
        }
        dot = warp_sum(dot);
        if (lane == l) p_mine = dot;
      }
    }
    float pv[LT], cv[LT + 1];
    cv[0] = 1.f;
#pragma unroll
    for (int l = 0; l < LT; ++l) {
      pv[l] = __shfl_sync(0xffffffffu, p_mine, l);
      const float q = __shfl_sync(0xffffffffu, q_mine, l);
      cv[l + 1] = cv[l] + fmaf(cv[l], pv[l], q);  // layers l >= L have p = q = 0: c stays
    }
    float al[LT];
    float t = 0.f, ds_mine = 0.f;
#pragma unroll
    for (int l = LT - 1; l >= 0; --l) {
      float ds = 0.f;
      if (l < L) {
        ds = a + t;
        t = fmaf(ds, pv[l], t);
      }
      al[l] = ds * cv[l];
      if (lane == l) ds_mine = ds;
    }
    Dacc += ds_mine;
    const float cL = cv[LT];
#pragma unroll
    for (int e = 0; e < E; ++e) dx[e] *= cL;
#pragma unroll
    for (int l = 0; l < LT; ++l) {
      if (l < L) {  // warp-uniform
        const float* wl = s_w + l * DP + lane * VEC;
#pragma unroll
        for (int i = 0; i < NPL; ++i) {
          const Pack<VEC> pw = lds_pack<VEC>(wl + i * 32 * VEC);
#pragma unroll
          for (int e = 0; e < VEC; ++e) {
            dx[i * VEC + e] = fmaf(al[l], pw.v[e], dx[i * VEC + e]);
            acc[l][i * VEC + e] = fmaf(al[l], x0[i * VEC + e], acc[l][i * VEC + e]);
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < NPL; ++i) {
      const int c = (i * 32 + lane) * VEC;
      if (c < d) st_pack<VEC>(dx0g + b * d + c, &dx[i * VEC]);
    }
  }
  // ---- the CTA's partials: warps in order, one quantity at a time through the (now idle) ring
  __syncthreads();
  float* comb = ring;  // [kCrossWarps][DP]
#pragma unroll
  for (int r = 0; r <= LT; ++r) {
    if (r <= L) {  // block-uniform
#pragma unroll
      for (int i = 0; i < NPL; ++i) {
        float4 v;
        if (r == 0) {
          v = make_float4(accdy[i * 4], accdy[i * 4 + 1], accdy[i * 4 + 2], accdy[i * 4 + 3]);
        } else {
          const int l = r > 0 ? r - 1 : 0;
          v = make_float4(acc[l][i * 4], acc[l][i * 4 + 1], acc[l][i * 4 + 2], acc[l][i * 4 + 3]);
        }
        *reinterpret_cast<float4*>(comb + wib * DP + (i * 32 + lane) * VEC) = v;
      }
      __syncthreads();
      for (int c = threadIdx.x; c < d; c += kCrossWarps * 32) {
        float tsum = 0.f;
#pragma unroll
        for (int w = 0; w < kCrossWarps; ++w) tsum += comb[w * DP + c];
        if (r == 0)
          dypart[(int64_t)blockIdx.x * d + c] = tsum;
        else
          dwpart[((int64_t)blockIdx.x * L + (r - 1)) * d + c] = tsum;
      }
      __syncthreads();
    }
  }
  sD[wib * 32 + lane] = Dacc;
  __syncthreads();
  if (threadIdx.x < L) {
    float tsum = 0.f;
#pragma unroll
    for (int w = 0; w < kCrossWarps; ++w) tsum += sD[w * 32 + threadIdx.x];
    Dpart[(int64_t)blockIdx.x * L + threadIdx.x] = tsum;
  }
}

template <int N, int T>
static void launch_ring(int grid, size_t smem, cudaStream_t st, const float* x0, const float* w, const float* b,
                        const float* dy, const float* p, int64_t B, int d, int L, int depth, float* dx0,
                        float* Dpart, float* dypart, float* dwpart) {
  if constexpr (4 * N * (T + 3) <= 184) {  // the register budget of one lane; other shapes take the tiled kernel
    cudaFuncSetAttribute(cross_bwd_ring_kernel<N, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cross_bwd_ring_kernel<N, T><<<grid, kCrossWarps * 32, smem, st>>>(x0, w, b, dy, p, B, d, L, depth, dx0, Dpart,
                                                                       dypart, dwpart);
  }
}

// Fixed-order combine of per-CTA partials: a CTA owns 8 columns; 32 "g-lanes" per column each sum
// every 32nd partial in order, then the 32 sums are added in lane order.
__global__ void __launch_bounds__(256)
cross_bwd_finish2_kernel(const float* __restrict__ wg, const float* __restrict__ bg,
                         const float* __restrict__ Dpart, const float* __restrict__ dypart,
                         const float* __restrict__ dwpart, int G1, int G2, int d, int L,
                         float* __restrict__ dw, float* __restrict__ db) {
  __shared__ float sDl[32];       // sum_b ds_l
  __shared__ float red[32][9];
  __shared__ float rows[33][8];   // row 0: sum dy; row 1+l: sum alpha_l x0
  const int cx = threadIdx.x & 7, gy = threadIdx.x >> 3;
  const int c = blockIdx.x * 8 + cx;
  {  // D_l: thread (l = gy, part = cx) sums every 8th partial, then the 8 parts in order
    float t = 0.f;
    if (gy < L)
      for (int g = cx; g < G1; g += 8) t += Dpart[(int64_t)g * L + gy];
    red[gy][cx] = t;
    __syncthreads();
    if (cx == 0) {
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) v += red[gy][k];
      sDl[gy] = v;
    }
    __syncthreads();
  }
  for (int r = 0; r <= L; ++r) {
    float t = 0.f;
    if (c < d) {
      if (r == 0) {
#pragma unroll 8
        for (int g = gy; g < G1; g += 32) t += __ldg(dypart + (int64_t)g * d + c);
      } else {
#pragma unroll 8
        for (int g = gy; g < G2; g += 32) t += __ldg(dwpart + ((int64_t)g * L + (r - 1)) * d + c);
      }
    }
    red[gy][cx] = t;
    __syncthreads();
    if (gy == 0) {
      float v = 0.f;
#pragma unroll
      for (int k = 0; k < 32; ++k) v += red[k][cx];
      rows[r][cx] = v;
    }
    __syncthreads();
  }
  if (gy != 0 || c >= d) return;
  // db_l = sum dy + sum_{j>l} w_j D_j ; walk l downwards carrying the tail
  float tail = 0.f;
  for (int l = L - 1; l >= 0; --l) {
    db[l * d + c] = rows[0][cx] + tail;
    tail = fmaf(wg[l * d + c], sDl[l], tail);
  }
  // dw_l = sum alpha_l x0 + beta_l D_l ; beta_l = sum_{j<l} b_j
  float beta = 0.f;
  for (int l = 0; l < L; ++l) {
    dw[l * d + c] = fmaf(beta, sDl[l], rows[1 + l][cx]);
    beta += bg[l * d + c];
  }
}

struct CrossShape {
  int vec, npl;
};
static bool cross_shape(int d, CrossShape& s) {
  if (d <= 0 || d > 1024) return false;
  if ((d & 3) == 0) {
    const int n = (d / 4 + 31) / 32;  // float4 per lane
    s.vec = 4;
    s.npl = n <= 6 ? n : 8;
    return true;
  }
  const int n = (d + 31) / 32;
  s.vec = 1;
  s.npl = n <= 1 ? 1 : n <= 2 ? 2 : n <= 4 ? 4 : n <= 8 ? 8 : n <= 16 ? 16 : 32;
  return true;
}

#define DIR_CROSS_DISPATCH(FN)                         \
  if (sh.vec == 4) {                                   \
    switch (sh.npl) {                                  \
      case 1: FN(4, 1); break;                         \
      case 2: FN(4, 2); break;                         \
      case 3: FN(4, 3); break;                         \
      case 4: FN(4, 4); break;                         \
      case 5: FN(4, 5); break;                         \
      case 6: FN(4, 6); break;                         \
      default: FN(4, 8); break;                        \
    }                                                  \
  } else {                                             \
    switch (sh.npl) {                                  \
      case 1: FN(1, 1); break;                         \
      case 2: FN(1, 2); break;                         \
      case 4: FN(1, 4); break;                         \
      case 8: FN(1, 8); break;                         \
      case 16: FN(1, 16); break;                       \
      default: FN(1, 32); break;                       \
    }                                                  \
  }

}  // namespace dir

extern "C" int dir_cross_fwd(const float* x0, const float* cross_w, const float* cross_b,
                             int64_t B, int d, int L, float* xL, float* s, dir_stream_t stream) {
  using namespace dir;
  CrossShape sh;
  if (B < 0 || L < 0 || L > 32 || !cross_shape(d, sh))
    return fail(DIR_EINVAL, "cross_fwd: need B >= 0, 0 <= L <= 32, 0 < d <= 1024");
  if (B == 0) return 0;
  if (!x0 || !xL || (L > 0 && (!cross_w || !cross_b)))
    return fail(DIR_EINVAL, "cross_fwd: null pointer");
  if (sh.vec == 4 && (!aligned16(x0) || !aligned16(xL) || !aligned16(cross_w) || !aligned16(cross_b)))
    return fail(DIR_EINVAL, "cross_fwd: 16-byte alignment required when d % 4 == 0");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // one warp per pair of samples; persistent beyond 4 CTAs per SM (each CTA recomputes beta_L, q_l)
  const int64_t want = (B + 2 * kCrossWarps - 1) / (2 * kCrossWarps);
  const unsigned grid = (unsigned)(want < (int64_t)kSMs * 2 ? want : (int64_t)kSMs * 2);
  // w staged in shared memory when it fits beside two resident CTAs per SM, else read through L1
#define DIR_FWD(V, N)                                                                               \
  {                                                                                                 \
    const size_t wbytes = (size_t)L * (V * N * 32) * 4;                                             \
    if (wbytes <= 64 * 1024) {                                                                      \
      cudaFuncSetAttribute(cross_fwd_kernel<V, N, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                           (int)wbytes);                                                            \
      cross_fwd_kernel<V, N, true><<<grid, kCrossWarps * 32, wbytes, st>>>(x0, cross_w, cross_b, B, d, \
                                                                           L, xL, s);               \
    } else {                                                                                        \
      cross_fwd_kernel<V, N, false><<<grid, kCrossWarps * 32, 0, st>>>(x0, cross_w, cross_b, B, d, L, \
                                                                       xL, s);                      \
    }                                                                                               \
  }
  DIR_CROSS_DISPATCH(DIR_FWD)
#undef DIR_FWD
  return launched("cross_fwd");
}

extern "C" size_t dir_cross_bwd_workspace_bytes(int64_t B, int d, int L) {
  if (B <= 0 || d <= 0 || L <= 0) return 256;
  return dir::cross_carve(nullptr, B, d, L).total;
}

extern "C" int dir_cross_bwd(const float* x0, const float* cross_w, const float* cross_b,
                             const float* dy, const float* s, int64_t B, int d, int L, float* dx0,
                             float* dw, float* db, void* workspace, size_t workspace_bytes,
                             dir_stream_t stream) {
  using namespace dir;
  CrossShape sh;
  if (B < 0 || L <= 0 || L > 32 || !cross_shape(d, sh))
    return fail(DIR_EINVAL, "cross_bwd: need B >= 0, 0 < L <= 32, 0 < d <= 1024");
  if (!dw || !db || (B > 0 && (!x0 || !cross_w || !cross_b || !dy || !dx0 || !workspace)))
    return fail(DIR_EINVAL, "cross_bwd: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (B == 0) {
    cudaMemsetAsync(dw, 0, (size_t)L * d * 4, st);
    cudaMemsetAsync(db, 0, (size_t)L * d * 4, st);
    return 0;
  }
  if (sh.vec == 4 && (!aligned16(x0) || !aligned16(dy) || !aligned16(dx0) || !aligned16(cross_w) ||
                      !aligned16(cross_b)))
    return fail(DIR_EINVAL, "cross_bwd: 16-byte alignment required when d % 4 == 0");
  CrossBwdWs w = cross_carve(workspace, B, d, L);
  if (workspace_bytes < w.total) return fail(DIR_ENOMEM, "cross_bwd: workspace too small");
  if (L <= 8 && sh.vec == 4) {
    // per-warp rings: needs the batch sums of one warp in registers and at least a two-slot ring in shared memory
    const int LT = (L + 1) & ~1;
    const size_t fixed = ((size_t)L * (4 * sh.npl * 32) + kCrossWarps * 32 + 32 + kCrossWarps) * 4;
    int depth = kRingMaxDepth;
    while (depth > 1 && fixed + (size_t)kCrossWarps * depth * 2 * d * 4 > 216 * 1024) --depth;
    if (4 * sh.npl * (LT + 3) <= 184 && depth >= 2) {
      const size_t ring_f = std::max((size_t)kCrossWarps * depth * 2 * d, (size_t)kCrossWarps * 4 * sh.npl * 32);
      const size_t smemr = fixed + ring_f * 4;
      const int64_t want = (B + kCrossWarps - 1) / kCrossWarps;
      // one CTA per SM, and never more CTAs than the workspace holds partials for (G1 = min(B / 16, two per SM))
      const int grid = (int)std::min<int64_t>(std::min<int64_t>(want, kSMs), w.G1);
#define DIR_BWDR(N, T)                                                                                   \
  if (sh.npl == N && LT == T)                                                                            \
    launch_ring<N, T>(grid, smemr, st, x0, cross_w, cross_b, dy, s, B, d, L, depth, dx0, w.Dpart, w.dypart, \
                      w.dwpart);
#define DIR_BWDR4(N) DIR_BWDR(N, 2) DIR_BWDR(N, 4) DIR_BWDR(N, 6) DIR_BWDR(N, 8)
      DIR_BWDR4(1) DIR_BWDR4(2) DIR_BWDR4(3) DIR_BWDR4(4) DIR_BWDR4(5) DIR_BWDR4(6) DIR_BWDR4(8)
#undef DIR_BWDR4
#undef DIR_BWDR
      cross_bwd_finish2_kernel<<<(d + 7) / 8, 256, 0, st>>>(cross_w, cross_b, w.Dpart, w.dypart, w.dwpart,
                                                             grid, grid, d, L, dw, db);
      return launched("cross_bwd", 2);
    }
  }
  if (L <= 8) {
    const size_t smem0 = ((size_t)2 * kTS * d + kTS * 8 + kCrossWarps * 32 + 32 + kCrossWarps) * 4;
#define DIR_BWDF(V, N)                                                                          \
  {                                                                                             \
    const size_t smemf = smem0 + (size_t)L * (V * N * 32) * 4;                                  \
    cudaFuncSetAttribute(cross_bwd_fused_kernel<V, N>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                         (int)smemf);                                                           \
    cross_bwd_fused_kernel<V, N><<<w.G1, kCrossWarps * 32, smemf, st>>>(                        \
        x0, cross_w, cross_b, dy, s, B, d, L, dx0, w.Dpart, w.dypart, w.dwpart);                \
  }
    DIR_CROSS_DISPATCH(DIR_BWDF)
#undef DIR_BWDF
    cross_bwd_finish2_kernel<<<(d + 7) / 8, 256, 0, st>>>(cross_w, cross_b, w.Dpart, w.dypart, w.dwpart,
                                                           w.G1, w.G2, d, L, dw, db);
    return launched("cross_bwd", 2);
  }
  const size_t smem1 = (size_t)kCrossWarps * (d + 32) * 4;
#define DIR_BWD(V, N)                                                                        \
  cross_bwd_sample_kernel<V, N><<<w.G1, kCrossWarps * 32, smem1, st>>>(                      \
      x0, cross_w, cross_b, dy, nullptr, B, d, L, dx0, w.alpha, w.Dpart, w.dypart)
  DIR_CROSS_DISPATCH(DIR_BWD)
#undef DIR_BWD
  cross_bwd_dw_kernel<<<w.G2, 256, kDwUnroll * 8 * 4, st>>>(x0, w.alpha, B, d, L, w.dwpart);
  cross_bwd_finish2_kernel<<<(d + 7) / 8, 256, 0, st>>>(cross_w, cross_b, w.Dpart, w.dypart, w.dwpart,
                                                         w.G1, w.G2, d, L, dw, db);
  return launched("cross_bwd", 3);
}
