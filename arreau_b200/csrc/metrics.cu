// Structural quality metrics of generated crystals (include/arreau_b200.h, "Beyond the reference"): volume, the exact
// minimum-image distance over distinct atom pairs, density and the number of distinct elements, one warp per crystal.
//
// Exactness of the minimum-image search.  The basis is first reduced (pairwise size reduction, below); L' = rows
// b1, b2, b3 of the reduced basis spans the same lattice.  For a pair, d = (f_j - f_i) L is shifted by the lattice
// vector that brings its reduced fractional coordinates t = d L'^-1 into [-0.5, 0.5]^3.  Pass 1 takes the 27 images
// t + k, k in {-1,0,1}^3, of every pair; their minimum over the crystal, R, bounds the true minimum from above.  An
// image with |(t + k) L'| <= R has |t_i + k_i| <= R |r_i| (r_i the columns of L'^-1), so |k_i| <= K_i =
// floor(1 + R |r_i|).  If every K_i <= 1, pass 1 was exact; otherwise pass 2 searches the box [-K, K] for every pair
// and sets ARREAU_METRICS_EXTENDED_SEARCH.
//
// Every output of a crystal depends only on that crystal: the pair-to-lane assignment depends on its atom count
// alone, the minimum is order-independent and the mass sum runs in atom order.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kMetricsWarps = 4;        // crystals per 128-thread CTA
constexpr int kReduceSweeps = 64;       // bound on the sweeps of the basis reduction
constexpr int kMaxSearch = 16;          // pass 2 searches at most [-16, 16] images per axis (ARREAU_METRICS_DEGENERATE)
constexpr double kAmuPerA3ToGPerCm3 = 1.66053906660;

__device__ __forceinline__ double dot3(const double (&a)[3], const double (&b)[3]) {
  return fma(a[0], b[0], fma(a[1], b[1], a[2] * b[2]));
}

__device__ __forceinline__ double warp_min(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ void cross3(const double (&a)[3], const double (&b)[3], double (&c)[3]) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}

// b_i -= rint(<b_i, b_j> / |b_j|^2) b_j; true if b_i changed.  Each change shortens b_i, so the sum of squared
// lengths falls strictly and the sweeps below end on a lattice; kReduceSweeps bounds them for any input.
__device__ __forceinline__ bool size_reduce(double (&bi)[3], const double (&bj)[3]) {
  const double q = rint(dot3(bi, bj) / dot3(bj, bj));
  if (q == 0.0 || !isfinite(q)) return false;
#pragma unroll
  for (int c = 0; c < 3; ++c) bi[c] = fma(-q, bj[c], bi[c]);
  return true;
}

// Calls f(i, j) once for every unordered pair i != j of an n-atom crystal, split over the 32 lanes of a warp by a
// rule that depends on n and the lane only.  Pairs (i, i + s mod n) for s = 1 .. (n - 1) / 2 cover each pair once
// for odd n; for even n the pairs (i, i + n / 2), i < n / 2, complete the set.
template <typename F>
__device__ __forceinline__ void for_each_pair(int n, int lane, F&& f) {
  const int64_t S = (n - 1) / 2;
  const int64_t total = (int64_t)n * S;
  if (lane < total) {
    int64_t s = 1 + lane / n;
    int i = lane % n;
    for (int64_t q = lane; q < total; q += 32) {
      int j = i + (int)s;
      if (j >= n) j -= n;
      f(i, j);
      i += 32;
      while (i >= n) {
        i -= n;
        ++s;
      }
    }
  }
  if ((n & 1) == 0)
    for (int i = lane; i < n / 2; i += 32) f(i, i + n / 2);
}

__global__ void __launch_bounds__(32 * kMetricsWarps) crystal_metrics_kernel(
    const double* __restrict__ frac, const double* __restrict__ lattice, const int64_t* __restrict__ atomic_numbers,
    const int32_t* __restrict__ atom_offset, int32_t N, int32_t G, const double* __restrict__ atomic_mass,
    int32_t max_z, double min_dist_threshold, double min_volume, double* __restrict__ volume_out,
    double* __restrict__ min_dist_out, double* __restrict__ density_out, int32_t* __restrict__ num_elements_out,
    int32_t* __restrict__ flags_out) {
  const int lane = threadIdx.x & 31;
  const int g = blockIdx.x * kMetricsWarps + (threadIdx.x >> 5);
  if (g >= G) return;
  const int a0 = atom_offset[g], a1 = atom_offset[g + 1];
  const bool bad_offsets = !(a0 >= 0 && a1 >= a0 && a1 <= N);
  const int n = bad_offsets ? 0 : a1 - a0;

  // ---- cell: every lane holds the lattice, its volume and the reduced basis ----
  double L[3][3];
  bool finite_cell = true;
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      L[r][c] = lattice[(int64_t)g * 9 + r * 3 + c];
      finite_cell = finite_cell && isfinite(L[r][c]);
    }
  double bc[3];
  cross3(L[1], L[2], bc);
  const double vol = fabs(dot3(L[0], bc));

  // ---- atoms: unknown elements, distinct known elements, mass in atom order, finite coordinates ----
  bool unknown = false, finite_frac = true;
  int distinct = 0;
  double mass = 0.0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    double m = 0.0;
    if (i < n) {
      const int64_t z = atomic_numbers[a0 + i];
      const bool known = z >= 0 && z <= max_z && atomic_mass[z] > 0.0;
      m = known ? atomic_mass[z] : nan("");
      unknown = unknown || !known;
      if (known) {
        bool first = true;
        for (int k = 0; k < i && first; ++k) first = atomic_numbers[a0 + k] != z;
        distinct += first;
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) finite_frac = finite_frac && isfinite(frac[(int64_t)(a0 + i) * 3 + c]);
    }
    const int cnt = min(32, n - base);
    for (int l = 0; l < cnt; ++l) mass += __shfl_sync(0xffffffffu, m, l);
  }
  unknown = __any_sync(0xffffffffu, unknown);
  finite_frac = __all_sync(0xffffffffu, finite_frac);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) distinct += __shfl_xor_sync(0xffffffffu, distinct, o);

  bool degenerate = bad_offsets || !finite_cell || !finite_frac || !(vol >= min_volume);
  bool extended = false;
  double dmin = degenerate ? nan("") : INFINITY;
  if (!degenerate && n >= 2) {
    double b[3][3];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) b[r][c] = L[r][c];
    for (int sweep = 0; sweep < kReduceSweeps; ++sweep) {
      bool changed = size_reduce(b[0], b[1]);
      changed |= size_reduce(b[0], b[2]);
      changed |= size_reduce(b[1], b[0]);
      changed |= size_reduce(b[1], b[2]);
      changed |= size_reduce(b[2], b[0]);
      changed |= size_reduce(b[2], b[1]);
      if (!changed) break;
    }
    // rows of (L'^-1)^T: t_i = <d, rc_i> with rc_i = (b_j x b_k) / det L'
    double rc[3][3];
    cross3(b[1], b[2], rc[0]);
    cross3(b[2], b[0], rc[1]);
    cross3(b[0], b[1], rc[2]);
    const double inv_det = 1.0 / dot3(b[0], rc[0]);
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) rc[r][c] *= inv_det;

    // d of pair (i, j) in the reduced cell, t in [-0.5, 0.5]^3
    auto wrapped = [&](int i, int j, double (&d)[3]) {
      double df[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) df[c] = __ldg(frac + (int64_t)(a0 + j) * 3 + c) - __ldg(frac + (int64_t)(a0 + i) * 3 + c);
#pragma unroll
      for (int c = 0; c < 3; ++c) d[c] = fma(df[0], L[0][c], fma(df[1], L[1][c], df[2] * L[2][c]));
      double s[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) s[r] = rint(dot3(d, rc[r]));
#pragma unroll
      for (int c = 0; c < 3; ++c) d[c] = fma(-s[0], b[0][c], fma(-s[1], b[1][c], fma(-s[2], b[2][c], d[c])));
    };

    double best = INFINITY;   // squared distance
    for_each_pair(n, lane, [&](int i, int j) {
      double d[3];
      wrapped(i, j, d);
#pragma unroll
      for (int ka = -1; ka <= 1; ++ka) {
        double u[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) u[c] = d[c] + ka * b[0][c];
#pragma unroll
        for (int kb = -1; kb <= 1; ++kb) {
          double v[3];
#pragma unroll
          for (int c = 0; c < 3; ++c) v[c] = u[c] + kb * b[1][c];
#pragma unroll
          for (int kc = -1; kc <= 1; ++kc) {
            double w[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) w[c] = v[c] + kc * b[2][c];
            best = fmin(best, dot3(w, w));
          }
        }
      }
    });
    best = warp_min(best);
    const double R = sqrt(best);
    double K[3];
#pragma unroll
    for (int r = 0; r < 3; ++r) K[r] = floor(1.0 + R * sqrt(dot3(rc[r], rc[r])));
    const double kmax = fmax(K[0], fmax(K[1], K[2]));
    if (!(kmax <= kMaxSearch)) {
      degenerate = true;      // also catches a non-finite R (coordinates too large for fp64)
      best = nan("");
    } else if (kmax > 1.0) {
      extended = true;
      const int K0 = (int)K[0], K1 = (int)K[1], K2 = (int)K[2];
      for_each_pair(n, lane, [&](int i, int j) {
        double d[3];
        wrapped(i, j, d);
        for (int ka = -K0; ka <= K0; ++ka) {
          double u[3];
#pragma unroll
          for (int c = 0; c < 3; ++c) u[c] = fma((double)ka, b[0][c], d[c]);
          for (int kb = -K1; kb <= K1; ++kb) {
            double v[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) v[c] = fma((double)kb, b[1][c], u[c]);
            for (int kc = -K2; kc <= K2; ++kc) {
              double w[3];
#pragma unroll
              for (int c = 0; c < 3; ++c) w[c] = fma((double)kc, b[2][c], v[c]);
              best = fmin(best, dot3(w, w));
            }
          }
        }
      });
      best = warp_min(best);
    }
    dmin = sqrt(best);
  }

  if (lane == 0) {
    volume_out[g] = vol;
    min_dist_out[g] = dmin;
    density_out[g] = mass * kAmuPerA3ToGPerCm3 / vol;
    num_elements_out[g] = distinct;
    int flags = 0;
    if (!degenerate && dmin >= min_dist_threshold) flags |= ARREAU_METRICS_VALID;
    if (unknown) flags |= ARREAU_METRICS_UNKNOWN_ELEMENT;
    if (degenerate) flags |= ARREAU_METRICS_DEGENERATE;
    if (extended) flags |= ARREAU_METRICS_EXTENDED_SEARCH;
    flags_out[g] = flags;
  }
}

}  // namespace

extern "C" int arreau_crystal_metrics(const double* frac, const double* lattice, const int64_t* atomic_numbers,
                                      const int32_t* atom_offset, int32_t num_atoms_total, int32_t num_crystals,
                                      const double* atomic_mass, int32_t max_z, double min_dist_threshold,
                                      double min_volume, double* volume, double* min_dist, double* density,
                                      int32_t* num_elements, int32_t* flags, void* stream) {
  if (num_crystals == 0) return ARREAU_OK;
  if (!lattice || !atom_offset || !atomic_mass || !volume || !min_dist || !density || !num_elements || !flags)
    return ARREAU_ERR_NULL;
  if (num_atoms_total > 0 && (!frac || !atomic_numbers)) return ARREAU_ERR_NULL;
  if (num_crystals < 0 || num_atoms_total < 0 || max_z < 0 || isnan(min_dist_threshold) || isnan(min_volume))
    return ARREAU_ERR_BAD_SHAPE;
  const unsigned blocks = (unsigned)((num_crystals + kMetricsWarps - 1) / kMetricsWarps);
  crystal_metrics_kernel<<<blocks, 32 * kMetricsWarps, 0, (cudaStream_t)stream>>>(
      frac, lattice, atomic_numbers, atom_offset, num_atoms_total, num_crystals, atomic_mass, max_z,
      min_dist_threshold, min_volume, volume, min_dist, density, num_elements, flags);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}
