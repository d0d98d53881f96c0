// Training-step kernels on the diffusion side (SURVEY 8a rows a19-a21), fp64 like the reference:
//   matrix_to_params            diffusion/lattice_helpers.py:16-35
//   VE_pbc.forward              diffusion/diffusion_helpers.py:43-63 (+ min_distance_sqr_pbc :254-325,
//                               cart_to_frac_coords :233-251)
//   D3PM.get_xt / q_sample      diffusion/d3pm.py:119-127,139-143
//   VP_lattice.forward          diffusion/diffusion_helpers.py:156-163
//   the three-term loss         diffusion/diffusion_loss.py:95-110,253-274, diffusion/d3pm.py:74-117,145-163
//                               and its gradient with respect to the network outputs
//   the same loss per crystal       for evaluation (no gradients): the per-atom terms of the training loss summed
//                                   over each crystal's own atoms
// The random draws are inputs (the reference's torch CPU stream is replayed by the host, or a device generator
// fills them); nothing here draws numbers.
#include "common.cuh"

namespace {

constexpr double kEps = 1e-6;   // diffusion/d3pm.py:23

__device__ __forceinline__ double remainder1(double a) {   // torch.remainder(a, 1.0)
  double m = fmod(a, 1.0);
  if (m != 0.0 && m < 0.0) m = __dadd_rn(m, 1.0);
  return m;
}

__global__ void matrix_to_params_kernel(const double* __restrict__ lattice, int G, double* __restrict__ lengths,
                                        double* __restrict__ angles) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const double* m = lattice + 9 * (size_t)g;
  double len[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    len[i] = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(m[3 * i], m[3 * i]), __dmul_rn(m[3 * i + 1], m[3 * i + 1])),
                            __dmul_rn(m[3 * i + 2], m[3 * i + 2])));
    lengths[3 * g + i] = len[i];
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    const double dot = __dadd_rn(__dadd_rn(__dmul_rn(m[3 * j], m[3 * k]), __dmul_rn(m[3 * j + 1], m[3 * k + 1])),
                                 __dmul_rn(m[3 * j + 2], m[3 * k + 2]));
    double v = __ddiv_rn(dot, __dmul_rn(len[j], len[k]));
    v = fmin(fmax(v, -1.0), 1.0);
    angles[3 * g + i] = acos(v);
  }
}

// one thread per atom
__global__ void ve_pbc_forward_kernel(const double* __restrict__ frac0, const double* __restrict__ eps,
                                      const int32_t* __restrict__ t_of_atom, const double* __restrict__ sigmas,
                                      const double* __restrict__ lattice, const int32_t* __restrict__ crystal_of_atom,
                                      int N, double* __restrict__ frac_noisy, double* __restrict__ target) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= N) return;
  const double* L = lattice + 9 * (size_t)crystal_of_atom[b];
  const double sig = sigmas[t_of_atom[b]];
  double f0[3], fn[3], pn[3], pp[3];
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    f0[d] = frac0[3 * (size_t)b + d];
    fn[d] = remainder1(__dadd_rn(f0[d], __dmul_rn(eps[3 * (size_t)b + d], sig)));   // helpers:45-46
    frac_noisy[3 * (size_t)b + d] = fn[d];
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {   // helpers:223-230
    pn[j] = __dadd_rn(__dadd_rn(__dmul_rn(fn[0], L[j]), __dmul_rn(fn[1], L[3 + j])), __dmul_rn(fn[2], L[6 + j]));
    pp[j] = __dadd_rn(__dadd_rn(__dmul_rn(f0[0], L[j]), __dmul_rn(f0[1], L[3 + j])), __dmul_rn(f0[2], L[6 + j]));
  }
  // helpers:283-309: v_k = pos1 - (pos2 + c_k @ L), first minimum of |v_k|^2 over the 27 cells in SUPERCELLS order
  double best = INFINITY, bv[3] = {0.0, 0.0, 0.0};
  for (int k = 0; k < 27; ++k) {
    const double c0 = (double)(k / 9 - 1), c1 = (double)((k / 3) % 3 - 1), c2 = (double)(k % 3 - 1);
    double v[3], d2 = 0.0;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double off = __dadd_rn(__dadd_rn(__dmul_rn(L[j], c0), __dmul_rn(L[3 + j], c1)), __dmul_rn(L[6 + j], c2));
      v[j] = __dadd_rn(pn[j], -__dadd_rn(pp[j], off));
    }
    d2 = __dadd_rn(__dadd_rn(__dmul_rn(v[0], v[0]), __dmul_rn(v[1], v[1])), __dmul_rn(v[2], v[2]));
    if (d2 < best) {
      best = d2;
      bv[0] = v[0]; bv[1] = v[1]; bv[2] = v[2];
    }
  }
  // helpers:233-251: frac = cart @ pinv(L)  (full-rank cells: the inverse), then % 1
  const double a = L[0], bb = L[1], c = L[2], d = L[3], e = L[4], f = L[5], gg = L[6], h = L[7], i = L[8];
  const double A = e * i - f * h, B = -(d * i - f * gg), C = d * h - e * gg;
  const double det = a * A + bb * B + c * C;
  const double inv[9] = {A / det, (c * h - bb * i) / det, (bb * f - c * e) / det,
                         B / det, (a * i - c * gg) / det, (c * d - a * f) / det,
                         C / det, (bb * gg - a * h) / det, (a * e - bb * d) / det};
#pragma unroll
  for (int j = 0; j < 3; ++j)
    target[3 * (size_t)b + j] = remainder1(bv[0] * inv[j] + bv[1] * inv[3 + j] + bv[2] * inv[6 + j]);
}

__global__ void vp_lattice_forward_kernel(const double* __restrict__ lengths, const double* __restrict__ eps,
                                          const int32_t* __restrict__ t_of_crystal, const float* __restrict__ alpha_bars,
                                          int G, double* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * G) return;
  const float ab = alpha_bars[t_of_crystal[idx / 3]];          // fp32 table (quirk B1)
  const double s1 = (double)sqrtf(ab), s2 = (double)sqrtf(1.0f - ab);
  out[idx] = __dadd_rn(__dmul_rn(s1, lengths[idx]), __dmul_rn(s2, eps[idx]));
}

// one warp per atom: argmax_d log(Qbar_t[x0, d] + eps) + gumbel(u[b, d]), first index on ties
__global__ void __launch_bounds__(256)
d3pm_q_sample_kernel(const int64_t* __restrict__ types0, const double* __restrict__ u, const int32_t* __restrict__ t_of_atom,
                     const double* __restrict__ q_keep, const double* __restrict__ q_to_mask, int N, int Z,
                     int64_t* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const int b = warp, x0 = (int)types0[b], t = t_of_atom[b], mask = Z - 1;
  const double keep = q_keep[t - 1], to_mask = q_to_mask[t - 1];
  double best = -INFINITY;
  int best_d = 0x7fffffff;
  for (int d = lane; d < Z; d += 32) {
    double p;
    if (x0 != mask) p = (d == x0) ? keep : (d == mask ? to_mask : 0.0);
    else p = (d == mask) ? 1.0 : 0.0;
    double noise = u[(size_t)b * Z + d];
    noise = fmin(fmax(noise, kEps), 1.0);
    const double val = log(p + kEps) - log(-log(noise));
    if (val > best || (val == best && d < best_d)) { best = val; best_d = d; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int od = __shfl_xor_sync(0xffffffffu, best_d, o);
    if (ob > best || (ob == best && od < best_d)) { best = ob; best_d = od; }
  }
  if (lane == 0) out[b] = (int64_t)best_d;
}

// ---- loss terms per atom + gradients w.r.t. the network outputs ---------------------------------------------
// posterior logits (d3pm.py:74-110) of a probability vector s over the mask chain, entry d held by (lane, r)
struct Posterior {
  double keep1, tomask1, qa, qb;
  int xt, mask, t;
};
__device__ __forceinline__ double post_logit(const Posterior& q, int d, double s_d, double s_nomask, double s_mask,
                                             double logit_d) {
  if (q.t == 1) return logit_d;
  double f1;
  if (q.xt != q.mask) f1 = (d == q.xt) ? q.keep1 : 0.0;
  else f1 = (d == q.mask) ? 1.0 : q.tomask1;
  const double f2 = (d != q.mask) ? s_d * q.qa : s_nomask * q.qb + s_mask;
  return log(f1 + kEps) + log(f2 + kEps);
}

constexpr int kPer = 4;   // Z <= 128

// kGrad = false (evaluation): the same per-atom terms with every gradient store compiled out
template <bool kGrad>
__global__ void __launch_bounds__(256)
atom_loss_kernel(const float* __restrict__ score, const float* __restrict__ logits, const double* __restrict__ target_eps,
                 const int64_t* __restrict__ types0, const int64_t* __restrict__ types_t,
                 const int32_t* __restrict__ t_of_atom, const double* __restrict__ q_keep,
                 const double* __restrict__ q_to_mask, double onestep_keep, double onestep_to_mask, int T, int N, int Z,
                 double hybrid_coeff, double* __restrict__ terms /* [3][N]: frac, vb, ce */, float* __restrict__ dscore,
                 float* __restrict__ dlogits) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const int b = warp;
  const double invN = 1.0 / (double)N;
  // wrapped squared error of the fractional score (diffusion_loss.py:95-110)
  {
    double w2 = 0.0;
    if (lane < 3) {
      const double delta = (double)score[3 * (size_t)b + lane] - target_eps[3 * (size_t)b + lane];
      double a = fmod(fabs(delta), 1.0);
      a = fmin(fmax(a, 0.0), 1.0);
      const double wdist = fmin(a, 1.0 - a);
      if constexpr (kGrad) {
        const double sgn = (double)((delta > 0.0) - (delta < 0.0));
        const double branch = (a < 1.0 - a) ? 1.0 : ((a > 1.0 - a) ? -1.0 : 0.0);
        dscore[3 * (size_t)b + lane] = (float)(2.0 * wdist * branch * sgn * invN);
      }
      w2 = wdist * wdist;
    }
    const double w0 = __shfl_sync(0xffffffffu, w2, 0), w1 = __shfl_sync(0xffffffffu, w2, 1),
                 w2b = __shfl_sync(0xffffffffu, w2, 2);
    if (lane == 0) terms[b] = (w0 + w1) + w2b;
  }
  __syncwarp();
  Posterior q;
  q.mask = Z - 1;
  q.t = t_of_atom[b];
  q.xt = (int)types_t[b];
  q.keep1 = onestep_keep;
  q.tomask1 = onestep_to_mask;
  const int qi = (q.t >= 2) ? (q.t - 2) : (T - 1);
  q.qa = q_keep[qi];
  q.qb = q_to_mask[qi];
  const int x0 = (int)types0[b];
  // softmax of the predicted logits
  double lg[kPer], s[kPer];
  double mx = -INFINITY, l_x0 = 0.0;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    lg[r] = d < Z ? (double)logits[(size_t)b * Z + d] : -INFINITY;
    mx = fmax(mx, lg[r]);
    if (d == x0) l_x0 = lg[r];
  }
  mx = warp_max(mx);
  double sum = 0.0;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    s[r] = (lane + 32 * r) < Z ? exp(lg[r] - mx) : 0.0;
    sum += s[r];
  }
  sum = warp_sum(sum);
  const double lse = mx + log(sum);
  l_x0 = warp_sum(l_x0);
  if (lane == 0) terms[2 * (size_t)N + b] = lse - l_x0;        // cross entropy (d3pm.py:161)
  double s_nomask = 0.0, s_mask = 0.0;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    s[r] /= sum;
    if (d < Z && d != q.mask) s_nomask += s[r];
    if (d == q.mask) s_mask = s[r];
  }
  s_nomask = warp_sum(s_nomask);
  s_mask = warp_sum(s_mask);
  // "true" posterior from the integer x0 (d3pm.py:81-84): softmax(log(onehot + eps))
  const double tz = (1.0 + kEps) + (double)(Z - 1) * kEps;
  const double s0_hit = (1.0 + kEps) / tz, s0_miss = kEps / tz;
  const double s0_mask = (x0 == q.mask) ? s0_hit : s0_miss;
  const double s0_nomask = (x0 == q.mask) ? (double)(Z - 1) * s0_miss : s0_hit + (double)(Z - 2) * s0_miss;
  double d1[kPer], d2[kPer];
  double m1 = -INFINITY, m2 = -INFINITY;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    if (d < Z) {
      const double s0 = (d == x0) ? s0_hit : s0_miss;
      d1[r] = post_logit(q, d, s0, s0_nomask, s0_mask, log(((d == x0) ? 1.0 : 0.0) + kEps)) + kEps;
      d2[r] = post_logit(q, d, s[r], s_nomask, s_mask, lg[r]) + kEps;
    } else {
      d1[r] = d2[r] = -INFINITY;
    }
    m1 = fmax(m1, d1[r]);
    m2 = fmax(m2, d2[r]);
  }
  m1 = warp_max(m1);
  m2 = warp_max(m2);
  double z1 = 0.0, z2 = 0.0;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    if (lane + 32 * r < Z) { z1 += exp(d1[r] - m1); z2 += exp(d2[r] - m2); }
  }
  z1 = warp_sum(z1);
  z2 = warp_sum(z2);
  const double lz1 = m1 + log(z1), lz2 = m2 + log(z2);
  double vb = 0.0;
  double gk[kPer];          // d vb_b / d d2_k = P2_k - P1_k
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    gk[r] = 0.0;
    if (lane + 32 * r < Z) {
      const double lp1 = d1[r] - lz1, lp2 = d2[r] - lz2;
      const double p1 = exp(lp1);
      vb += p1 * (lp1 - lp2);
      gk[r] = exp(lp2) - p1;
    }
  }
  vb = warp_sum(vb);
  if (lane == 0) terms[(size_t)N + b] = vb;
  if constexpr (!kGrad) return;
  // gradient w.r.t. the logits
  const double cv = hybrid_coeff * invN;
  double dl[kPer];
  if (q.t == 1) {
#pragma unroll
    for (int r = 0; r < kPer; ++r) dl[r] = cv * gk[r];
  } else {
    // through f2 = s Qbar: ds_c = g_c qa / (f2_c + eps) + [c != mask] g_mask qb / (f2_mask + eps); mask row: g_mask / (..)
    const double f2_mask = s_nomask * q.qb + s_mask;
    double gmask = 0.0;
#pragma unroll
    for (int r = 0; r < kPer; ++r)
      if (lane + 32 * r == q.mask) gmask = gk[r] / (f2_mask + kEps);
    gmask = warp_sum(gmask);
    double ds[kPer], dot = 0.0;
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
      const int d = lane + 32 * r;
      ds[r] = 0.0;
      if (d < Z) {
        if (d != q.mask) ds[r] = gk[r] * q.qa / (s[r] * q.qa + kEps) + gmask * q.qb;
        else ds[r] = gmask;
        dot += s[r] * ds[r];
      }
    }
    dot = warp_sum(dot);
#pragma unroll
    for (int r = 0; r < kPer; ++r) dl[r] = cv * s[r] * (ds[r] - dot);
  }
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    if (d < Z) dlogits[(size_t)b * Z + d] = (float)(dl[r] + (s[r] - ((d == x0) ? 1.0 : 0.0)) * invN);
  }
}

// single block: fixed-order sums -> out[5] = {loss, e_frac, vb, ce, e_lat}; also dlen0
__global__ void __launch_bounds__(256)
loss_finish_kernel(const double* __restrict__ terms, const float* __restrict__ len0, const double* __restrict__ lengths,
                   const int32_t* __restrict__ atom_offset, int N, int G, double hybrid_coeff, double* __restrict__ out,
                   float* __restrict__ dlen0) {
  __shared__ double sh[4][256];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < N; i += 256) {
    acc[0] += terms[i];
    acc[1] += terms[(size_t)N + i];
    acc[2] += terms[2 * (size_t)N + i];
  }
  for (int i = threadIdx.x; i < 3 * G; i += 256) {
    const int g = i / 3;
    const double n = (double)(atom_offset[g + 1] - atom_offset[g]);
    const double diff = (double)len0[i] - lengths[i] / n;        // diffusion_loss.py:262-265
    acc[3] += diff * diff;
    dlen0[i] = (float)(2.0 * diff / (3.0 * (double)G));
  }
  for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] = acc[k];
  __syncthreads();
  for (int stride = 128; stride > 0; stride >>= 1) {
    if (threadIdx.x < stride)
      for (int k = 0; k < 4; ++k) sh[k][threadIdx.x] += sh[k][threadIdx.x + stride];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const double e_frac = sh[0][0] / (double)N, vb = sh[1][0] / (double)N, ce = sh[2][0] / (double)N;
    const double e_lat = sh[3][0] / (3.0 * (double)G);
    out[0] = e_frac + (vb * hybrid_coeff + ce) + e_lat;
    out[1] = e_frac; out[2] = vb; out[3] = ce; out[4] = e_lat;
  }
}

// one thread per crystal: sums over its own atoms in atom order, so a crystal's four numbers do not depend on which
// other crystals share the batch.  out[G][4] = {frac, vb, ce, sum_d (len0 - lengths / n)^2}
__global__ void crystal_loss_kernel(const double* __restrict__ terms, const float* __restrict__ len0,
                                    const double* __restrict__ lengths, const int32_t* __restrict__ atom_offset, int N,
                                    int G, double* __restrict__ out) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const int lo = atom_offset[g], hi = atom_offset[g + 1];
  double s0 = 0.0, s1 = 0.0, s2 = 0.0;
  for (int b = lo; b < hi; ++b) {
    s0 += terms[b];
    s1 += terms[(size_t)N + b];
    s2 += terms[2 * (size_t)N + b];
  }
  const double n = (double)(hi - lo);
  double lat = 0.0;
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const double diff = (double)len0[3 * g + d] - lengths[3 * g + d] / n;        // diffusion_loss.py:262-265
    lat += diff * diff;
  }
  out[4 * (size_t)g] = s0;
  out[4 * (size_t)g + 1] = s1;
  out[4 * (size_t)g + 2] = s2;
  out[4 * (size_t)g + 3] = lat;
}

// torch.optim.Adam step (diffusion.py:161-210: two weight-decay groups, L2 decay folded into the gradient) with the
// trainer's global-norm clip (main_diffusion.py:297, clip_grad_norm_: coef = min(1, max_norm / (norm + 1e-6))) read
// from the device so that the step never synchronises with the host.  With `ema`, the exponential moving average of
// the weights is updated from the new parameter in the same pass (the NeMo EMAOptimizer rule, applied after the inner
// step): ema = decay * ema + (1 - decay) * p_new; the parameter arithmetic is the same with or without it.
__global__ void __launch_bounds__(256)
adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                 const uint8_t* __restrict__ decay_mask, long long n, float lr, float beta1, float beta2, float eps,
                 float weight_decay, float bias_c1, float bias_c2_sqrt, float max_grad_norm,
                 const double* __restrict__ grad_moments, float* __restrict__ ema, float ema_decay,
                 float ema_one_minus_decay) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float coef = 1.0f;
  if (grad_moments && max_grad_norm > 0.f) {
    const float norm = (float)sqrt(grad_moments[1]);
    coef = fminf(max_grad_norm / (norm + 1e-6f), 1.0f);
  }
  float gi = g[i] * coef;
  const float pi = p[i];
  if (decay_mask && decay_mask[i]) gi = fmaf(weight_decay, pi, gi);
  const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
  const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / bias_c2_sqrt + eps;
  const float p_new = pi - (lr / bias_c1) * (mi / denom);
  p[i] = p_new;
  if (ema) ema[i] = fmaf(ema_one_minus_decay, p_new, ema_decay * ema[i]);
}

}  // namespace

extern "C" int arreau_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                                const uint8_t* decay_mask, int64_t n, double lr, double beta1, double beta2, double eps,
                                double weight_decay, int64_t step, double max_grad_norm, const double* grad_moments,
                                float* ema, double ema_decay, void* stream) {
  if (n == 0) return ARREAU_OK;
  if (!params || !grads || !exp_avg || !exp_avg_sq) return ARREAU_ERR_NULL;
  if (n < 0 || step < 1) return ARREAU_ERR_BAD_SHAPE;
  if (ema && !(ema_decay >= 0.0 && ema_decay <= 1.0)) return ARREAU_ERR_BAD_SHAPE;
  const double c1 = 1.0 - pow(beta1, (double)step), c2 = 1.0 - pow(beta2, (double)step);
  adam_step_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      params, grads, exp_avg, exp_avg_sq, decay_mask, n, (float)lr, (float)beta1, (float)beta2, (float)eps,
      (float)weight_decay, (float)c1, (float)sqrt(c2), (float)max_grad_norm, grad_moments, ema, (float)ema_decay,
      (float)(1.0 - ema_decay));
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_matrix_to_params(const double* lattice, int32_t G, double* lengths, double* angles, void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lattice || !lengths || !angles) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  matrix_to_params_kernel<<<(G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(lattice, G, lengths, angles);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_ve_pbc_forward(const double* frac0, const double* eps, const int32_t* t_of_atom,
                                     const double* ve_sigmas, const double* lattice, const int32_t* crystal_of_atom,
                                     int32_t N, double* frac_noisy, double* target_eps, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!frac0 || !eps || !t_of_atom || !ve_sigmas || !lattice || !crystal_of_atom || !frac_noisy || !target_eps)
    return ARREAU_ERR_NULL;
  if (N < 0) return ARREAU_ERR_BAD_SHAPE;
  ve_pbc_forward_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(frac0, eps, t_of_atom, ve_sigmas, lattice,
                                                                          crystal_of_atom, N, frac_noisy, target_eps);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_vp_lattice_forward(const double* lengths, const double* eps, const int32_t* t_of_crystal,
                                         const float* vp_alpha_bars, int32_t G, double* noisy_lengths, void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !eps || !t_of_crystal || !vp_alpha_bars || !noisy_lengths) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  vp_lattice_forward_kernel<<<(3 * G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(lengths, eps, t_of_crystal,
                                                                                  vp_alpha_bars, G, noisy_lengths);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_d3pm_q_sample(const int64_t* types0, const double* u, const int32_t* t_of_atom, const double* q_keep,
                                    const double* q_to_mask, int32_t N, int32_t Z, int64_t* types_t, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!types0 || !u || !t_of_atom || !q_keep || !q_to_mask || !types_t) return ARREAU_ERR_NULL;
  if (N < 0 || Z <= 1) return ARREAU_ERR_BAD_SHAPE;
  const long long threads = (long long)N * 32;
  d3pm_q_sample_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(types0, u, t_of_atom, q_keep,
                                                                                           q_to_mask, N, Z, types_t);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_training_loss(const float* score, const float* logits, const float* len0, const double* target_eps,
                                    const int64_t* types0, const int64_t* types_t, const int32_t* t_of_atom,
                                    const double* lengths, const int32_t* atom_offset, const double* q_keep,
                                    const double* q_to_mask, double onestep_keep, double onestep_to_mask,
                                    int32_t num_steps, int32_t N, int32_t G, int32_t Z, double hybrid_coeff,
                                    double* terms_scratch, double* loss_out, float* dscore, float* dlogits, float* dlen0,
                                    void* stream) {
  if (!score || !logits || !len0 || !target_eps || !types0 || !types_t || !t_of_atom || !lengths || !atom_offset ||
      !q_keep || !q_to_mask || !terms_scratch || !loss_out || !dscore || !dlogits || !dlen0)
    return ARREAU_ERR_NULL;
  if (N <= 0 || G <= 0 || Z <= 1 || Z > 128 || num_steps <= 0) return ARREAU_ERR_BAD_SHAPE;
  const long long threads = (long long)N * 32;
  atom_loss_kernel<true><<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      score, logits, target_eps, types0, types_t, t_of_atom, q_keep, q_to_mask, onestep_keep, onestep_to_mask, num_steps,
      N, Z, hybrid_coeff, terms_scratch, dscore, dlogits);
  CUDA_LAUNCH_CHECK();
  loss_finish_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(terms_scratch, len0, lengths, atom_offset, N, G, hybrid_coeff,
                                                          loss_out, dlen0);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_eval_loss(const float* score, const float* logits, const float* len0, const double* target_eps,
                                const int64_t* types0, const int64_t* types_t, const int32_t* t_of_atom,
                                const double* lengths, const int32_t* atom_offset, const double* q_keep,
                                const double* q_to_mask, double onestep_keep, double onestep_to_mask, int32_t num_steps,
                                int32_t N, int32_t G, int32_t Z, double* terms_scratch, double* per_crystal,
                                void* stream) {
  if (!score || !logits || !len0 || !target_eps || !types0 || !types_t || !t_of_atom || !lengths || !atom_offset ||
      !q_keep || !q_to_mask || !terms_scratch || !per_crystal)
    return ARREAU_ERR_NULL;
  if (N <= 0 || G <= 0 || Z <= 1 || Z > 128 || num_steps <= 0) return ARREAU_ERR_BAD_SHAPE;
  const long long threads = (long long)N * 32;
  atom_loss_kernel<false><<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      score, logits, target_eps, types0, types_t, t_of_atom, q_keep, q_to_mask, onestep_keep, onestep_to_mask, num_steps,
      N, Z, 0.0, terms_scratch, nullptr, nullptr);
  CUDA_LAUNCH_CHECK();
  crystal_loss_kernel<<<(G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(terms_scratch, len0, lengths, atom_offset, N, G,
                                                                         per_crystal);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}
