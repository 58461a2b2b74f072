// Row-update arithmetic shared by every kernel that applies a de-duplicated gradient to a table row
// or a first-order weight (embed_bwd.cu, shard_peer.cu): [TF] SparseApplyAdagrad / ScatterSub /
// SparseApplyFtrl behind optimizer.minimize, models/DeepFM/deepFM.py:230-241 (SURVEY.md row A9).
#pragma once
#include "common.cuh"

namespace dir {

// The linear scope (first-order weights) has an optimizer of its own in the reference
// (linear_optimizer='Ftrl', models/DeepFM/deepFM.py:58, 236-241).
struct LinOpt {
  int opt;      // DIR_OPT_SGD | DIR_OPT_ADAGRAD | DIR_OPT_FTRL
  float lr;
  float l1, l2; // Ftrl regularisation strengths
  float* z;     // Ftrl 'linear' slot, same stride as the weights
};

// Row update with the de-duplicated gradient: a = acc + g*g; T = T - (lr*g) * rsqrt(a)
// ([TF] SparseApplyAdagrad, no epsilon; Eigen evaluates it as lr * g * rsqrt(a) as well).  rsqrtf
// is MUFU.RSQ (<= 2 ulp): an IEEE divide + square root per component made this line a quarter of
// all instructions the kernel issued (profiles/r01_reduce_v1_source.txt).
__device__ __forceinline__ float upd(float t, float g, float lr, float& a, bool adagrad) {
  if (adagrad) {
    a = __fadd_rn(a, __fmul_rn(g, g));
    return __fsub_rn(t, __fmul_rn(__fmul_rn(lr, g), rsqrtf(a)));
  }
  return __fsub_rn(t, __fmul_rn(lr, g));
}

// [TF] SparseApplyProximalAdagrad (tf.train.ProximalAdagradOptimizer, the reference's dnn_optimizer in
// models/ESMM/train.py:137-139), accumulator starting at 0.1:
//   a += g^2;  eta = lr * rsqrt(a);  p = t - g * eta
//   t = sign(p) * max(|p| - eta * l1, 0) / (1 + l2 * eta)        (l1 = 0: t = p / (1 + l2 * eta))
__device__ __forceinline__ float upd_prox(float t, float g, float lr, float& a, float l1, float l2) {
  a = __fadd_rn(a, __fmul_rn(g, g));
  const float eta = __fmul_rn(lr, rsqrtf(a));
  const float p = __fsub_rn(t, __fmul_rn(g, eta));
  const float den = __fadd_rn(1.f, __fmul_rn(l2, eta));
  if (l1 > 0.f) return __fdiv_rn(copysignf(fmaxf(__fsub_rn(fabsf(p), __fmul_rn(eta, l1)), 0.f), p), den);
  return __fdiv_rn(p, den);
}
// the rule of a table row: SGD / Adagrad (upd) or ProximalAdagrad
struct RowRule {
  int opt;
  float lr, l1, l2;
};
__device__ __forceinline__ float upd_rule(float t, float g, float& a, const RowRule& r) {
  if (r.opt == DIR_OPT_PROXIMAL_ADAGRAD) return upd_prox(t, g, r.lr, a, r.l1, r.l2);
  return upd(t, g, r.lr, a, r.opt == DIR_OPT_ADAGRAD);
}

// One first-order weight with its de-duplicated gradient g.  Ftrl is [TF] SparseApplyFtrl with
// learning_rate_power = -0.5 and no l2 shrinkage (tf.train.FtrlOptimizer defaults):
//   n' = n + g^2;  sigma = (sqrt(n') - sqrt(n)) / lr;  z += g - sigma*w
//   w  = |z| > l1 ? (sign(z)*l1 - z) / (sqrt(n')/lr + 2*l2) : 0
__device__ __forceinline__ void lin_apply(const LinOpt& o, float* wp, float* np, float* zp, float w,
                                          float n, float z, float g) {
  if (o.opt == DIR_OPT_FTRL) {
    const float nn = __fadd_rn(n, __fmul_rn(g, g));
    const float rn = __fsqrt_rn(nn);
    const float sigma = __fdiv_rn(__fsub_rn(rn, __fsqrt_rn(n)), o.lr);
    z = __fsub_rn(__fadd_rn(z, g), __fmul_rn(sigma, w));
    const float quad = __fadd_rn(__fdiv_rn(rn, o.lr), __fmul_rn(2.f, o.l2));
    *wp = fabsf(z) > o.l1 ? __fdiv_rn(__fsub_rn(copysignf(o.l1, z), z), quad) : 0.f;
    *np = nn;
    *zp = z;
    return;
  }
  if (o.opt == DIR_OPT_PROXIMAL_ADAGRAD) {
    *wp = upd_prox(w, g, o.lr, n, o.l1, o.l2);
    *np = n;
    return;
  }
  const bool adagrad = o.opt == DIR_OPT_ADAGRAD;
  *wp = upd(w, g, o.lr, n, adagrad);
  if (adagrad) *np = n;
}
// loads for lin_apply (what each optimizer keeps per weight)
__device__ __forceinline__ void lin_load(const LinOpt& o, const float* lin_accum, int64_t off, float& n, float& z) {
  n = o.opt != DIR_OPT_SGD ? lin_accum[off] : 0.f;
  z = o.opt == DIR_OPT_FTRL ? o.z[off] : 0.f;
}

// dir_field_sqnorms' partials: [F][kClipSlices][2] doubles (sum of squares of G, of g1), one slice per CTA of the
// norm pass (clip.cu).  Read by every apply that scales a column's gradient by its clip_by_norm factor.
constexpr int kClipSlices = 16;
constexpr int kClipMaxFields = 1024;

// Per column f < F: its first row and the clip_by_norm denominators max(||G_f||, clip), max(||g1_f||, clip), from the
// partials summed in a fixed order (the same factor in every CTA).  Block-strided; the caller synchronises.
__device__ __forceinline__ void clip_denominators(const double* __restrict__ part, const int64_t* __restrict__ field_offset,
                                                  int F, float clip, int64_t* s_off, float* s_den, float* s_den1) {
  for (int f = threadIdx.x; f < F; f += blockDim.x) {
    s_off[f] = field_offset[f];
    double a = 0.0, b = 0.0;
    for (int s = 0; s < kClipSlices; ++s) {
      a += part[((int64_t)f * kClipSlices + s) * 2];
      b += part[((int64_t)f * kClipSlices + s) * 2 + 1];
    }
    s_den[f] = fmaxf((float)sqrt(a), clip);
    s_den1[f] = fmaxf((float)sqrt(b), clip);
  }
}

// [TF] clip_by_norm: values * clip_norm / max(l2norm, clip_norm)
__device__ __forceinline__ float clip1(float g, float clip, float denom) { return __fdiv_rn(__fmul_rn(g, clip), denom); }

// The linear scope's optimizer: the caller's dir_linear_opt, or the tables' optimizer and rate.
inline int resolve_lin(const char* what, const dir_linear_opt* in, int optimizer, float lr, const float* lin,
                       const float* lin_accum, LinOpt& out) {
  out = LinOpt{optimizer, lr, 0.f, 0.f, nullptr};
  if (in != nullptr) out = LinOpt{in->optimizer, in->lr, in->l1, in->l2, in->z};
  if (out.opt != DIR_OPT_SGD && out.opt != DIR_OPT_ADAGRAD && out.opt != DIR_OPT_FTRL &&
      out.opt != DIR_OPT_PROXIMAL_ADAGRAD)
    return fail(DIR_EINVAL, "%s: unknown linear optimizer", what);
  if (lin != nullptr) {
    if (out.opt != DIR_OPT_SGD && !lin_accum)
      return fail(DIR_EINVAL, "%s: Adagrad / ProximalAdagrad / Ftrl on the linear weights need lin_accum", what);
    if (out.opt == DIR_OPT_PROXIMAL_ADAGRAD && (out.l1 < 0.f || out.l2 < 0.f))
      return fail(DIR_EINVAL, "%s: l1, l2 must be >= 0", what);
    if (out.opt == DIR_OPT_FTRL && (!out.z || !(out.lr > 0.f) || out.l1 < 0.f || out.l2 < 0.f))
      return fail(DIR_EINVAL, "%s: Ftrl needs z, lr > 0 and l1, l2 >= 0", what);
  }
  return 0;
}

}  // namespace dir
