// K9 (feature assembly) and K8 (per-step update) -- the fp64 diffusion state side of the step.
//
// Everything here is tiny and HBM-bound; it is kept in fp64 because the reference keeps its
// state (frac, lengths, lattice, positions) in fp64 and the radius graph thresholds depend on it.
#include "common.cuh"

namespace {

constexpr double kPi = 3.141592653589793;   // np.pi
constexpr double kD3pmEps = 1e-6;           // diffusion/d3pm.py:23

// diffusion/lattice_helpers.py:69-105
__global__ void lattice_from_params_kernel(const double* __restrict__ lengths, const double* __restrict__ angles,
                                           int G, double* __restrict__ lattice) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const double a = lengths[3 * g], b = lengths[3 * g + 1], c = lengths[3 * g + 2];
  const double al = angles[3 * g], be = angles[3 * g + 1], ga = angles[3 * g + 2];
  const double ca = cos(al), cb = cos(be), cg = cos(ga);
  const double sa = sin(al), sb = sin(be);
  double val = __ddiv_rn(__dadd_rn(__dmul_rn(ca, cb), -cg), __dmul_rn(sa, sb));
  val = fmin(fmax(val, -1.0), 1.0);   // abs_cap (:79-82); NaN propagates like torch.clamp
  if (val != val) val = val;
  const double gs = acos(val);
  double* L = lattice + 9 * (size_t)g;
  L[0] = __dmul_rn(a, sb);
  L[1] = 0.0;
  L[2] = __dmul_rn(a, cb);
  L[3] = __dmul_rn(__dmul_rn(-b, sa), cos(gs));
  L[4] = __dmul_rn(__dmul_rn(b, sa), sin(gs));
  L[5] = __dmul_rn(b, ca);
  L[6] = 0.0;
  L[7] = 0.0;
  L[8] = c;
}

// lattice_helpers.py:85-96 with the angle factors [sin b, cos b, sin a, cos g*, sin g*, cos a] given
__global__ void lattice_from_trig_kernel(const double* __restrict__ lengths, const double* __restrict__ trig, int G,
                                         double* __restrict__ lattice) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= G) return;
  const double a = lengths[3 * g], b = lengths[3 * g + 1], c = lengths[3 * g + 2];
  const double* f = trig + 6 * (size_t)g;
  double* L = lattice + 9 * (size_t)g;
  L[0] = __dmul_rn(a, f[0]);
  L[1] = 0.0;
  L[2] = __dmul_rn(a, f[1]);
  L[3] = __dmul_rn(__dmul_rn(-b, f[2]), f[3]);
  L[4] = __dmul_rn(__dmul_rn(b, f[2]), f[4]);
  L[5] = __dmul_rn(b, f[5]);
  L[6] = 0.0;
  L[7] = 0.0;
  L[8] = c;
}

// diffusion/diffusion_helpers.py:223-230: pos_j = sum_i frac_i * L[i][j]  (einsum "bi,bij->bj")
__global__ void frac_to_cart_kernel(const double* __restrict__ frac, const double* __restrict__ lattice,
                                    const int32_t* __restrict__ crystal_of_atom, int N, double* __restrict__ pos) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= N) return;
  const double* L = lattice + 9 * (size_t)crystal_of_atom[b];
  const double f0 = frac[3 * b], f1 = frac[3 * b + 1], f2 = frac[3 * b + 2];
#pragma unroll
  for (int j = 0; j < 3; ++j)
    pos[3 * b + j] = __dadd_rn(__dadd_rn(__dmul_rn(f0, L[j]), __dmul_rn(f1, L[3 + j])), __dmul_rn(f2, L[6 + j]));
}

// diffusion/diffusion_loss.py:124-158: one warp per atom writes its F = Z + 2*emb + 10 scalars
// and its 4 vector channels.
__global__ void __launch_bounds__(256)
assemble_features_kernel(const double* __restrict__ frac, const int64_t* __restrict__ types,
                         const double* __restrict__ lengths, const double* __restrict__ angles,
                         const double* __restrict__ lattice, const int32_t* __restrict__ atom_offset,
                         const int32_t* __restrict__ crystal_of_atom, const int32_t* __restrict__ t_of_atom,
                         int t_scalar, const double* __restrict__ vp_betas, const double* __restrict__ fourier_w,
                         int emb, int N, int Z, float* __restrict__ x, float* __restrict__ vec) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const int b = warp, g = crystal_of_atom[b];
  const int F = Z + 2 * emb + 10;
  float* xr = x + (size_t)b * F;
  const int ty = (int)types[b];
  for (int z = lane; z < Z; z += 32) xr[z] = (z == ty) ? 1.0f : 0.0f;
  const int t = t_of_atom ? t_of_atom[b] : t_scalar;
  const double beta = vp_betas[t];                     // diffusion_loss.py:126
  for (int k = lane; k < emb; k += 32) {
    // helpers:24: x * w * 2 * np.pi, left to right
    const double xp = __dmul_rn(__dmul_rn(__dmul_rn(beta, fourier_w[k]), 2.0), kPi);
    double s, c;
    sincos(xp, &s, &c);
    xr[Z + k] = (float)s;
    xr[Z + emb + k] = (float)c;
  }
  if (lane < 10) {
    const double n = (double)(atom_offset[g + 1] - atom_offset[g]);
    double v;
    if (lane == 0) v = n;
    else if (lane < 4) v = lengths[3 * g + lane - 1];
    else if (lane < 7) v = angles[3 * g + lane - 4];
    else v = fabs(__ddiv_rn(lengths[3 * g + lane - 7], n));
    xr[Z + 2 * emb + lane] = (float)v;
  }
  if (lane < 12) {
    const double v = lane < 3 ? frac[3 * (size_t)b + lane] : lattice[9 * (size_t)g + lane - 3];
    vec[(size_t)b * 12 + lane] = (float)v;
  }
}

// diffusion/diffusion_helpers.py:185-199
//
// kKnown: a crystal g with known_crystal[g] != 0 has known lengths l0 = known_lengths[g] (structure-conditioned
// sampling, RePaint replacement).  Its reverse update is discarded and replaced by a draw of the forward process at the
// new level, q(x_{t-1} | l0) = sqrt(abar[t-1]) l0 + sqrt(1 - abar[t-1]) z with the step's own noise z and the fp32
// abar table -- the arithmetic of vp_lattice_forward_kernel, so the two are bit-identical -- and l0 itself at t == 1.
// The instance without it compiles to the code it had before the condition existed.
template <bool kKnown>
__global__ void vp_lattice_reverse_kernel(const double* lengths, const float* __restrict__ len0,
                                          const int32_t* __restrict__ atom_offset, const double* __restrict__ z,
                                          int t, double cx0, double cxt, double denom, double var, int G,
                                          double* out, const double* __restrict__ dyn,   // out may alias lengths
                                          const int32_t* __restrict__ known_crystal,
                                          const double* __restrict__ known_lengths,
                                          const float* __restrict__ alpha_bars) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * G) return;
  if (dyn) {      // replayable step: {t, cx0, cxt, denom, var} of the current replay live in device memory
    t = (int)dyn[0]; cx0 = dyn[1]; cxt = dyn[2]; denom = dyn[3]; var = dyn[4];
  }
  const int g = idx / 3;
  if constexpr (kKnown) {
    if (known_crystal[g]) {
      const double l0 = known_lengths[idx];
      if (t >= 2) {
        const float ab = alpha_bars[t - 1];                           // fp32 table (quirk B1)
        const double s1 = (double)sqrtf(ab), s2 = (double)sqrtf(1.0f - ab);
        out[idx] = __dadd_rn(__dmul_rn(s1, l0), __dmul_rn(s2, z[idx]));
      } else {
        out[idx] = l0;
      }
      return;
    }
  }
  const double n = (double)(atom_offset[g + 1] - atom_offset[g]);
  const double pred = __dmul_rn((double)len0[idx], n);            // diffusion_loss.py:338
  const double mean = __ddiv_rn(__dadd_rn(__dmul_rn(cx0, pred), __dmul_rn(cxt, lengths[idx])), denom);
  const double zz = (t > 1) ? z[idx] : 0.0;
  out[idx] = __dadd_rn(mean, __dmul_rn(var, zz));                 // `variance * z`: quirk B5
}

__device__ __forceinline__ double torch_remainder1(double a) {
  // torch.remainder(a, 1.0) on CPU: fmod, then shift into the divisor's sign
  double m = fmod(a, 1.0);
  if (m != 0.0 && m < 0.0) m = __dadd_rn(m, 1.0);
  return m;
}

// diffusion/diffusion_helpers.py:65-81
//
// kKnown: an atom b with known_atom[b] != 0 has a known position x0 = known_frac[b] in [0,1)^3.  Its reverse update is
// replaced by q(x_{t-1} | x0) = (x0 + z sigma[t-1]) mod 1 with the step's own noise z -- the arithmetic of
// ve_pbc_forward_kernel at level t-1, so the two are bit-identical -- and by x0 itself at t == 1.
template <bool kKnown>
__global__ void ve_pbc_reverse_kernel(const double* frac, const float* __restrict__ score,
                                      const double* __restrict__ z, const int32_t* __restrict__ t_of_atom,
                                      int t_scalar, const double* __restrict__ sigmas, int N,
                                      double* out,   // out may alias frac
                                      const int32_t* __restrict__ known_atom, const double* __restrict__ known_frac) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * N) return;
  const int t = t_of_atom ? t_of_atom[idx / 3] : t_scalar;
  if constexpr (kKnown) {
    if (known_atom[idx / 3]) {
      const double x0 = known_frac[idx];
      out[idx] = t >= 2 ? torch_remainder1(__dadd_rn(x0, __dmul_rn(z[idx], sigmas[t - 1]))) : x0;
      return;
    }
  }
  const double s = sigmas[t];
  const double a = (t == 0) ? 0.0 : sigmas[t - 1];
  const double s2 = __dmul_rn(s, s), a2 = __dmul_rn(a, a);
  const double d = __dadd_rn(s2, -a2);
  const double mean = __dadd_rn(frac[idx], -__dmul_rn((double)score[idx], d));
  const double rnd = __dmul_rn(sqrt(__ddiv_rn(__dmul_rn(a2, d), s2)), z[idx]);
  out[idx] = torch_remainder1(__dadd_rn(mean, rnd));
}

// diffusion/d3pm.py:74-110,198-215 for the mask-absorbing chain; one warp per atom.
//
// kAllowed: the states an atom may take are restricted to its crystal's set A, bit d of allowed[4 g + d / 32] for
// state d of crystal g = crystal_of_atom[b] (bits at d >= Z are ignored; a set with no bit below Z counts as every
// state, so no input leaves an atom without a candidate).  For that atom:
//   1. the x0 probabilities are the softmax of the logits over A: a state outside A has probability 0 (this is what
//      sum_nomask, p_mask and f2 see);
//   2. the argmax runs over A plus the mask state Z-1 at t >= 2 (the mask absorbs: a masked atom may stay masked), and
//      over A alone at t == 1.  The exclusion is explicit: a state outside A still has the finite posterior
//      log(f1 + eps) + log(0 + eps), which the Gumbel noise could lift above the others;
//   3. with every state in A the result is bit-identical to the unconstrained kernel (the arithmetic is the same).
// The unconstrained instantiation compiles to the code it had before the constraint existed.
//
// kKnown: an atom b with known_atom[b] != 0 keeps its state at every step, t == 1 included (structure-conditioned
// sampling: its type is part of the known structure).  Without the override the t == 1 argmax would sample it from the
// logits, and at t >= 2 the finite log(0 + eps) term would still let it flip.
template <bool kAllowed, bool kKnown>
__global__ void __launch_bounds__(256)
d3pm_reverse_kernel(const int64_t* types, const float* __restrict__ logits,
                    const double* __restrict__ u, const int32_t* __restrict__ t_of_atom, int t_scalar,
                    const double* __restrict__ q_keep, const double* __restrict__ q_to_mask,
                    double onestep_keep, double onestep_to_mask, int T, int N, int Z,
                    int64_t* out,   // out may alias types
                    const int32_t* __restrict__ crystal_of_atom, const uint32_t* __restrict__ allowed,
                    const int32_t* __restrict__ known_atom) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const int b = warp;
  if constexpr (kKnown) {
    if (known_atom[b]) {
      if (lane == 0) out[b] = types[b];
      return;
    }
  }
  const int t = t_of_atom ? t_of_atom[b] : t_scalar;
  const int xt = (int)types[b];
  const int mask = Z - 1;
  constexpr int kPer = 4;   // Z <= 128: lane's state d = lane + 32 r is bit `lane` of the crystal's mask word r
  uint32_t in_set = 0xfu;   // bit r: state lane + 32 r is in A
  if constexpr (kAllowed) {
    const uint32_t* w = allowed + (size_t)kPer * crystal_of_atom[b];
    uint32_t any = 0, mine = 0;
#pragma unroll
    for (int r = 0; r < kPer; ++r) {
      const int lo = 32 * r;   // keep the bits of states d < Z only
      const uint32_t valid = Z - lo >= 32 ? 0xffffffffu : (Z - lo <= 0 ? 0u : (1u << (Z - lo)) - 1u);
      const uint32_t word = w[r];
      any |= word & valid;
      mine |= ((word >> lane) & 1u) << r;
    }
    if (any) in_set = mine;
  }
  double lg[kPer], p[kPer];
  double mx = -INFINITY;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    lg[r] = (d < Z && ((in_set >> r) & 1u)) ? (double)logits[(size_t)b * Z + d] : -INFINITY;
    mx = fmax(mx, lg[r]);
  }
  mx = warp_max(mx);
  double sum = 0.0, sum_nomask = 0.0;
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    p[r] = d < Z ? exp(lg[r] - mx) : 0.0;
    sum += p[r];
  }
  sum = warp_sum(sum);
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    p[r] = p[r] / sum;
    if (d < Z && d != mask) sum_nomask += p[r];
  }
  sum_nomask = warp_sum(sum_nomask);
  double p_mask = 0.0;
  {
    const int r = mask >> 5;
    double v = 0.0;
#pragma unroll
    for (int rr = 0; rr < kPer; ++rr)
      if (rr == r) v = p[rr];
    p_mask = __shfl_sync(0xffffffffu, v, mask & 31);
  }
  // cumulative matrix Qbar = q_mats[t-2] (d3pm.py:101); t == 1 wraps to index -1 but is masked out (B11)
  const int qi = (t >= 2) ? (t - 2) : (T - 1);
  const double qa = q_keep[qi], qb = q_to_mask[qi];
  // (t != 1).float() -> fp32: 0.2f + 0.8f == 1.0f, 0.2f + 0 == 0.2f, promoted to fp64 (d3pm.py:209-210)
  const double scale = (t != 1) ? 1.0 : (double)0.2f;
  double best = -INFINITY;
  int best_d = 0x7fffffff;
  // q_one_step_transposed[t-1, x_t, d] = Q[d, x_t] only takes two values per atom: their logs are evaluated once
  // (same log on the same doubles as the per-element form: identical bits)
  const double f1_hit = (xt != mask) ? onestep_keep : 1.0, f1_miss = (xt != mask) ? 0.0 : onestep_to_mask;
  const double lf1_hit = log(f1_hit + kD3pmEps), lf1_miss = log(f1_miss + kD3pmEps);
#pragma unroll
  for (int r = 0; r < kPer; ++r) {
    const int d = lane + 32 * r;
    if (d >= Z) continue;
    if (kAllowed && !((in_set >> r) & 1u) && (t == 1 || d != mask)) continue;   // rule 2
    double lp;
    if (t == 1) {
      lp = lg[r];
    } else {
      const bool hit = (xt != mask) ? (d == xt) : (d == mask);
      double f2;   // sum_c softmax_c * Qbar[c, d]
      if (d != mask) f2 = p[r] * qa;
      else f2 = sum_nomask * qb + p_mask;
      lp = (hit ? lf1_hit : lf1_miss) + log(f2 + kD3pmEps);
    }
    double noise = u[(size_t)b * Z + d];
    noise = fmin(fmax(noise, kD3pmEps), 1.0);
    const double gumbel = -log(-log(noise));
    const double val = lp + gumbel * scale;
    if (val > best || (val == best && d < best_d)) {
      best = val;
      best_d = d;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int od = __shfl_xor_sync(0xffffffffu, best_d, o);
    if (ob > best || (ob == best && od < best_d)) {
      best = ob;
      best_d = od;
    }
  }
  if (lane == 0) out[b] = (int64_t)best_d;
}

}  // namespace

extern "C" int arreau_lattice_from_params(const double* lengths, const double* angles, int32_t G,
                                          double* lattice, void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !angles || !lattice) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  lattice_from_params_kernel<<<(G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(lengths, angles, G, lattice);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_lattice_from_trig(const double* lengths, const double* trig, int32_t G, double* lattice,
                                        void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !trig || !lattice) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  lattice_from_trig_kernel<<<(G + 127) / 128, 128, 0, (cudaStream_t)stream>>>(lengths, trig, G, lattice);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_frac_to_cart(const double* frac, const double* lattice, const int32_t* crystal_of_atom,
                                   int32_t N, double* pos, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!frac || !lattice || !crystal_of_atom || !pos) return ARREAU_ERR_NULL;
  if (N < 0) return ARREAU_ERR_BAD_SHAPE;
  frac_to_cart_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(frac, lattice, crystal_of_atom, N, pos);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_assemble_features(const double* frac, const int64_t* types, const double* lengths,
                                        const double* angles, const double* lattice, const int32_t* atom_offset,
                                        const int32_t* crystal_of_atom, const int32_t* t_of_atom, int32_t t,
                                        const double* vp_betas, const double* fourier_w, int32_t emb, int32_t N,
                                        int32_t G, int32_t Z, float* x, float* vec, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!frac || !types || !lengths || !angles || !lattice || !atom_offset || !crystal_of_atom || !vp_betas ||
      !fourier_w || !x || !vec)
    return ARREAU_ERR_NULL;
  if (N < 0 || G <= 0 || Z <= 0 || emb <= 0) return ARREAU_ERR_BAD_SHAPE;
  const long long threads = (long long)N * 32;
  assemble_features_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      frac, types, lengths, angles, lattice, atom_offset, crystal_of_atom, t_of_atom, t, vp_betas, fourier_w, emb,
      N, Z, x, vec);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

namespace {

int launch_vp_lattice_reverse(const double* lengths, const float* len0, const int32_t* atom_offset, const double* z,
                              int32_t t, double cx0, double cxt, double denom, double var, int32_t G, const double* dyn,
                              const int32_t* known_crystal, const double* known_lengths, const float* alpha_bars,
                              double* lengths_out, void* stream) {
  const unsigned blocks = (unsigned)((3 * G + 127) / 128);
  if (known_crystal)
    vp_lattice_reverse_kernel<true><<<blocks, 128, 0, (cudaStream_t)stream>>>(
        lengths, len0, atom_offset, z, t, cx0, cxt, denom, var, G, lengths_out, dyn, known_crystal, known_lengths,
        alpha_bars);
  else
    vp_lattice_reverse_kernel<false><<<blocks, 128, 0, (cudaStream_t)stream>>>(
        lengths, len0, atom_offset, z, t, cx0, cxt, denom, var, G, lengths_out, dyn, nullptr, nullptr, nullptr);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

int launch_ve_pbc_reverse(const double* frac, const float* score, const double* z, const int32_t* t_of_atom, int32_t t,
                          const double* ve_sigmas, int32_t N, const int32_t* known_atom, const double* known_frac,
                          double* frac_out, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!frac || !score || !z || !ve_sigmas || !frac_out) return ARREAU_ERR_NULL;
  if (N < 0) return ARREAU_ERR_BAD_SHAPE;
  const unsigned blocks = (unsigned)((3 * N + 255) / 256);
  if (known_atom)
    ve_pbc_reverse_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(frac, score, z, t_of_atom, t, ve_sigmas, N,
                                                                         frac_out, known_atom, known_frac);
  else
    ve_pbc_reverse_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(frac, score, z, t_of_atom, t, ve_sigmas, N,
                                                                          frac_out, nullptr, nullptr);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

}  // namespace

extern "C" int arreau_vp_lattice_reverse(const double* lengths, const float* len0, const int32_t* atom_offset,
                                         const double* z, int32_t t, double cx0, double cxt, double denom,
                                         double var, int32_t G, double* lengths_out, void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !len0 || !atom_offset || !lengths_out || (t > 1 && !z)) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  return launch_vp_lattice_reverse(lengths, len0, atom_offset, z, t, cx0, cxt, denom, var, G, nullptr, nullptr, nullptr,
                                   nullptr, lengths_out, stream);
}

extern "C" int arreau_vp_lattice_reverse_known(const double* lengths, const float* len0, const int32_t* atom_offset,
                                               const double* z, int32_t t, double cx0, double cxt, double denom,
                                               double var, int32_t G, const int32_t* known_crystal,
                                               const double* known_lengths, const float* vp_alpha_bars,
                                               double* lengths_out, void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !len0 || !atom_offset || !lengths_out || (t > 1 && !z)) return ARREAU_ERR_NULL;
  if (!known_crystal || !known_lengths || !vp_alpha_bars) return ARREAU_ERR_NULL;
  if (G < 0) return ARREAU_ERR_BAD_SHAPE;
  return launch_vp_lattice_reverse(lengths, len0, atom_offset, z, t, cx0, cxt, denom, var, G, nullptr, known_crystal,
                                   known_lengths, vp_alpha_bars, lengths_out, stream);
}

// the same with the timestep and the four posterior coefficients read from device memory (arreau_denoise_step_replay);
// known_crystal NULL: no known lattice
int arreau_vp_lattice_reverse_dyn(const double* lengths, const float* len0, const int32_t* atom_offset, const double* z,
                                  const double* dyn, int32_t G, const int32_t* known_crystal,
                                  const double* known_lengths, const float* vp_alpha_bars, double* lengths_out,
                                  void* stream) {
  if (G == 0) return ARREAU_OK;
  if (!lengths || !len0 || !atom_offset || !lengths_out || !z || !dyn) return ARREAU_ERR_NULL;
  if (known_crystal && (!known_lengths || !vp_alpha_bars)) return ARREAU_ERR_NULL;
  return launch_vp_lattice_reverse(lengths, len0, atom_offset, z, 0, 0.0, 0.0, 1.0, 0.0, G, dyn, known_crystal,
                                   known_lengths, vp_alpha_bars, lengths_out, stream);
}

extern "C" int arreau_ve_pbc_reverse(const double* frac, const float* score, const double* z,
                                     const int32_t* t_of_atom, int32_t t, const double* ve_sigmas, int32_t N,
                                     double* frac_out, void* stream) {
  return launch_ve_pbc_reverse(frac, score, z, t_of_atom, t, ve_sigmas, N, nullptr, nullptr, frac_out, stream);
}

extern "C" int arreau_ve_pbc_reverse_known(const double* frac, const float* score, const double* z,
                                           const int32_t* t_of_atom, int32_t t, const double* ve_sigmas, int32_t N,
                                           const int32_t* known_atom, const double* known_frac, double* frac_out,
                                           void* stream) {
  if (N != 0 && (!known_atom || !known_frac)) return ARREAU_ERR_NULL;
  return launch_ve_pbc_reverse(frac, score, z, t_of_atom, t, ve_sigmas, N, known_atom, known_frac, frac_out, stream);
}

namespace {

int launch_d3pm_reverse(const int64_t* types, const float* logits, const double* u, const int32_t* t_of_atom, int32_t t,
                        const double* q_keep, const double* q_to_mask, double onestep_keep, double onestep_to_mask,
                        int32_t num_steps, int32_t N, int32_t Z, const int32_t* crystal_of_atom, const uint32_t* allowed,
                        const int32_t* known_atom, int64_t* types_out, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!types || !logits || !u || !q_keep || !q_to_mask || !types_out) return ARREAU_ERR_NULL;
  if (N < 0 || Z <= 1 || Z > 128 || num_steps <= 0) return ARREAU_ERR_BAD_SHAPE;
  const long long threads = (long long)N * 32;
  const unsigned blocks = (unsigned)((threads + 255) / 256);
  cudaStream_t s = (cudaStream_t)stream;
#define ARREAU_D3PM_LAUNCH(A, K)                                                                                      \
  d3pm_reverse_kernel<A, K><<<blocks, 256, 0, s>>>(types, logits, u, t_of_atom, t, q_keep, q_to_mask, onestep_keep, \
                                                   onestep_to_mask, num_steps, N, Z, types_out, crystal_of_atom,     \
                                                   allowed, known_atom)
  if (allowed && known_atom) ARREAU_D3PM_LAUNCH(true, true);
  else if (allowed) ARREAU_D3PM_LAUNCH(true, false);
  else if (known_atom) ARREAU_D3PM_LAUNCH(false, true);
  else ARREAU_D3PM_LAUNCH(false, false);
#undef ARREAU_D3PM_LAUNCH
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

}  // namespace

extern "C" int arreau_d3pm_reverse(const int64_t* types, const float* logits, const double* u,
                                   const int32_t* t_of_atom, int32_t t, const double* q_keep,
                                   const double* q_to_mask, double onestep_keep, double onestep_to_mask,
                                   int32_t num_steps, int32_t N, int32_t Z, int64_t* types_out, void* stream) {
  return launch_d3pm_reverse(types, logits, u, t_of_atom, t, q_keep, q_to_mask, onestep_keep, onestep_to_mask,
                             num_steps, N, Z, nullptr, nullptr, nullptr, types_out, stream);
}

extern "C" int arreau_d3pm_reverse_allowed(const int64_t* types, const float* logits, const double* u,
                                           const int32_t* t_of_atom, int32_t t, const double* q_keep,
                                           const double* q_to_mask, double onestep_keep, double onestep_to_mask,
                                           int32_t num_steps, int32_t N, int32_t Z, const int32_t* crystal_of_atom,
                                           const uint32_t* allowed, int64_t* types_out, void* stream) {
  if (N != 0 && (!crystal_of_atom || !allowed)) return ARREAU_ERR_NULL;
  return launch_d3pm_reverse(types, logits, u, t_of_atom, t, q_keep, q_to_mask, onestep_keep, onestep_to_mask,
                             num_steps, N, Z, crystal_of_atom, allowed, nullptr, types_out, stream);
}

extern "C" int arreau_d3pm_reverse_known(const int64_t* types, const float* logits, const double* u,
                                         const int32_t* t_of_atom, int32_t t, const double* q_keep,
                                         const double* q_to_mask, double onestep_keep, double onestep_to_mask,
                                         int32_t num_steps, int32_t N, int32_t Z, const int32_t* crystal_of_atom,
                                         const uint32_t* allowed, const int32_t* known_atom, int64_t* types_out,
                                         void* stream) {
  if (N != 0 && (!known_atom || (allowed && !crystal_of_atom))) return ARREAU_ERR_NULL;
  return launch_d3pm_reverse(types, logits, u, t_of_atom, t, q_keep, q_to_mask, onestep_keep, onestep_to_mask,
                             num_steps, N, Z, crystal_of_atom, allowed, known_atom, types_out, stream);
}
