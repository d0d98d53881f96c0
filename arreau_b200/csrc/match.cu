// Paired structure matcher (include/arreau_b200.h, "Beyond the reference"): generated crystal g against source
// crystal g, as pymatgen's StructureMatcher(stol, ltol, angle_tol, scale=True, attempt_supercell=False,
// primitive_cell=False).get_rms_dist(generated, source) computes it; one warp per pair.  Each step mirrors a pymatgen
// function:
//   reduction       Structure.get_reduced_structure("niggli") -> Lattice.get_niggli_reduced_lattice: Krivy-Gruber
//                   with e = 1e-5 V^(1/3) on the LLL basis (Lattice._calculate_lll, delta = 0.75).  The integer
//                   transform is kept and the coordinates are re-expressed in it, so no find_mapping is needed;
//   scale           StructureMatcher._preprocess: ratio = (V2 / V1)^(1/6), L1 *= ratio, L2 /= ratio;
//   mappings        Lattice.find_all_mappings + StructureMatcher._get_lattices: triples of s1's lattice vectors in
//                   the three length bands of s2 with s2's angles, |det| = 1 (no supercells);
//   per mapping     StructureMatcher._get_supercells (average lattice from the mean parameters,
//                   Lattice.from_parameters) and _strict_match (normalisation, frac_tol);
//   translations    StructureMatcher._get_mask: anchored on the first s2 site of the rarest element;
//   prefilter       StructureMatcher._cmp_fstruct -> coord_cython.is_coord_subset_pbc;
//   assignment      StructureMatcher._cart_dists -> coord_cython.pbc_shortest_vectors (LLL basis of the average
//                   lattice, lll_frac_tol, 27 images of the mod-1 coordinates) + LinearAssignment, solved here as
//                   a shortest-augmenting-path (Jonker-Volgenant / Hungarian) per element block with the
//                   inadmissible pairs excluded (pymatgen prices them at 1e20; a translation without a complete
//                   matching is rejected here);
//   result          the smallest rms = |dist| / sqrt(n) over every mapping and translation (first one on ties).
//
// Fit (arreau_structure_fit_pairs, structure_match_kernel<true>): StructureMatcher(stol, ltol, angle_tol, scale=True,
// attempt_supercell=False, primitive_cell=False).fit(a, b), i.e. _match(..., use_rms=False, break_on_match=True), on
// pair p = crystal index1[p] of set 1 (a, whose lattice is mapped, as struct1) and crystal index2[p] of set 2 (b).  The
// pipeline above is unchanged; a candidate's value is max(dist) instead of the rms, the pair is matched iff some
// candidate has max(dist) < stol, and the search stops at the first such candidate in the fixed enumeration order
// (mappings by band index ia, ib, ic, then translations), leaving every loop warp-uniformly.  Outputs: max_dist (the
// first value below stol, else the smallest found, NaN without a candidate), num_mappings (the mappings visited: all
// of them when not matched) and flags.  Fit-matched implies rms-matched (rms <= max on the same candidate), not the
// converse.  The uniqueness / novelty bookkeeping on top of it (inference/structure_match.py) is pymatgen's
// group_structures on crystals with the same multiset of Z: with primitive_cell=False and no supercells, fit never
// holds between different atom counts.  The kFit = false instance compiles to the same SASS as before the template.
//
// Layout.  Atoms are sorted by Z within each crystal (the host sorts, stably), so the element blocks of the two
// crystals coincide when their compositions do, and atom k of either crystal has the same element.  A warp holds its
// pair's coordinates in shared memory; per-pair and per-mapping lattice work (LLL, Niggli, the average lattice) is
// scalar and runs redundantly in every lane.  The lattice points of the three bands are enumerated lane-parallel in a
// fixed order (ballot-compacted), the mappings are evaluated on the fly in band order, the prefilter runs lane-parallel
// over s2 sites with an early exit, and the assignment gives the lanes the columns (s1 sites): a row's costs are
// computed when it enters the alternating tree and the warp argmin takes the lowest column on ties.  There are no
// atomics, and every reduction order depends on the pair's atom count only, so a pair's outputs depend only on that
// pair, bit for bit.
#include <math.h>

#include "common.cuh"

namespace {

constexpr int kMaxAtoms = 256;        // ARREAU_MATCH_TOO_LARGE above
constexpr int kBandCap = 128;         // lattice points per length band (ARREAU_MATCH_SEARCH_LIMIT above)
constexpr int kMaxSteps = 255;        // enumeration box half-width per axis (ARREAU_MATCH_SEARCH_LIMIT above)
constexpr int kLllIters = 1000;       // bounds of the reduction loops (ARREAU_MATCH_DEGENERATE when reached)
constexpr int kNiggliIters = 100;     // pymatgen's bound
constexpr double kMinVolume = 0.1;    // A^3

struct PairSmem {
  double f2[kMaxAtoms][3];            // s2 in its Niggli basis, [0, 1)
  double fc1[kMaxAtoms][3];           // s1 in the mapped basis, [0, 1)
  double lf1[kMaxAtoms][3];           // fc1 in the LLL basis of the average lattice, [0, 1)
  double lf2[kMaxAtoms][3];           // translated f2 in that basis, [0, 1)
  double u[kMaxAtoms + 1], v[kMaxAtoms + 1], minv[kMaxAtoms + 1];   // assignment duals and slacks (1-based)
  double im[27][3];                   // the 27 images (-1, 0, 1)^3 in the LLL basis, Cartesian
  int16_t p[kMaxAtoms + 1], way[kMaxAtoms + 1];
  int16_t row_of[kMaxAtoms];          // matched s2 site of every s1 site (whole crystal)
  uint8_t used[kMaxAtoms + 1];
  int32_t band[3][kBandCap];          // packed integer coordinates of the band points
  uint32_t mask[3][kBandCap][kBandCap / 32];   // angle tests: alpha (b, c), beta (a, c), gamma (a, b)
};

__device__ __forceinline__ double dot3(const double* a, const double* b) {
  return fma(a[0], b[0], fma(a[1], b[1], a[2] * b[2]));
}

__device__ __forceinline__ void cross3(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}

__device__ __forceinline__ double det3(const double (&m)[3][3]) {
  double c[3];
  cross3(m[1], m[2], c);
  return dot3(m[0], c);
}

__device__ __forceinline__ double wrap01(double x) { return x - floor(x); }

// x @ S (row vector times matrix)
__device__ __forceinline__ void vecmat(const double* x, const double (&S)[3][3], double* y) {
#pragma unroll
  for (int c = 0; c < 3; ++c) y[c] = fma(x[0], S[0][c], fma(x[1], S[1][c], x[2] * S[2][c]));
}

// inverse of an integer matrix with |det| = 1, exact: the adjugate over the determinant
__device__ void int_inverse(const double (&S)[3][3], double (&R)[3][3]) {
  const double d = det3(S);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int j1 = (j + 1) % 3, j2 = (j + 2) % 3, i1 = (i + 1) % 3, i2 = (i + 2) % 3;
      R[i][j] = (S[j1][i1] * S[j2][i2] - S[j1][i2] * S[j2][i1]) / d;
    }
}

// lengths of the columns of A^-1 (pymatgen's reciprocal_lattice.abc / 2 pi)
__device__ void recip_lengths(const double (&A)[3][3], double* r) {
  const double d = det3(A);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double c[3];
    cross3(A[(i + 1) % 3], A[(i + 2) % 3], c);
    r[i] = sqrt(dot3(c, c)) / fabs(d);
  }
}

// lengths and angles (degrees) of the rows of M, as pymatgen's Lattice.parameters
__device__ void lattice_params(const double (&M)[3][3], double* p) {
#pragma unroll
  for (int i = 0; i < 3; ++i) p[i] = sqrt(dot3(M[i], M[i]));
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const int j = (d + 1) % 3, k = (d + 2) % 3;
    p[3 + d] = acos(fmin(1.0, fmax(-1.0, dot3(M[j], M[k]) / (p[j] * p[k])))) * 180.0 / M_PI;
  }
}

// pymatgen Lattice.from_parameters (vesta = False)
__device__ void lattice_from_params(const double* p, double (&A)[3][3]) {
  const double al = p[3] * (M_PI / 180.0), be = p[4] * (M_PI / 180.0), ga = p[5] * (M_PI / 180.0);
  const double ca = cos(al), cb = cos(be), cg = cos(ga), sa = sin(al), sb = sin(be);
  const double gs = acos(fmin(1.0, fmax(-1.0, (ca * cb - cg) / (sa * sb))));
  A[0][0] = p[0] * sb;        A[0][1] = 0.0;              A[0][2] = p[0] * cb;
  A[1][0] = -p[1] * sa * cos(gs); A[1][1] = p[1] * sa * sin(gs); A[1][2] = p[1] * ca;
  A[2][0] = 0.0;              A[2][1] = 0.0;              A[2][2] = p[2];
}

// The three reduction routines below stay out of line: inlined into structure_match_kernel, the -O3 build (CUDA 12.9,
// sm_100a) returned failed reductions for ordinary cells that the same code reduces when it is compiled out of line,
// with -G, or for the host.
//
// pymatgen Lattice._calculate_lll on the rows of a (in place); map: reduced = map @ input.  False if it did not end.
__device__ __noinline__ bool lll_reduce(double (&a)[3][3], double (&map)[3][3]) {
  constexpr double delta = 0.75;
  double b[3][3], u[3][3] = {}, m[3];
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int c = 0; c < 3; ++c) map[i][c] = i == c ? 1.0 : 0.0;
#pragma unroll
  for (int c = 0; c < 3; ++c) b[0][c] = a[0][c];
  m[0] = dot3(b[0], b[0]);
#pragma unroll
  for (int i = 1; i < 3; ++i) {
    double s[3] = {0.0, 0.0, 0.0};
#pragma unroll
    for (int j = 0; j < i; ++j) {
      u[i][j] = dot3(a[i], b[j]) / m[j];
#pragma unroll
      for (int c = 0; c < 3; ++c) s[c] = fma(b[j][c], u[i][j], s[c]);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) b[i][c] = a[i][c] - s[c];
    m[i] = dot3(b[i], b[i]);
  }
  int k = 2;
  for (int it = 0; k <= 3; ++it) {
    if (it >= kLllIters) return false;
    for (int i = k - 1; i > 0; --i) {
      const double q = rint(u[k - 1][i - 1]);
      if (q != 0.0) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          a[k - 1][c] -= q * a[i - 1][c];
          map[k - 1][c] -= q * map[i - 1][c];
        }
        for (int j = 0; j < i - 1; ++j) u[k - 1][j] -= q * u[i - 1][j];
        u[k - 1][i - 1] -= q;
      }
    }
    const double mu = u[k - 1][k - 2];
    if (dot3(b[k - 1], b[k - 1]) >= (delta - mu * mu) * dot3(b[k - 2], b[k - 2])) {
      ++k;
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const double t = a[k - 1][c];
        a[k - 1][c] = a[k - 2][c];
        a[k - 2][c] = t;
        const double tm = map[k - 1][c];
        map[k - 1][c] = map[k - 2][c];
        map[k - 2][c] = tm;
      }
      for (int s = k - 2; s <= k - 1; ++s) {
        double acc[3] = {0.0, 0.0, 0.0};
        for (int j = 0; j < s; ++j) {
          u[s][j] = dot3(a[s], b[j]) / m[j];
#pragma unroll
          for (int c = 0; c < 3; ++c) acc[c] = fma(b[j][c], u[s][j], acc[c]);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) b[s][c] = a[s][c] - acc[c];
        m[s] = dot3(b[s], b[s]);
      }
      if (k > 2) {
        --k;
      } else {
        for (int r = k; r < 3; ++r)
          for (int j = k - 2; j < k; ++j) u[r][j] = dot3(a[r], b[j]) / m[j];
      }
    }
  }
  return true;
}

__device__ __forceinline__ void g6(const double (&b)[3][3], double& A, double& B, double& C, double& E, double& N,
                                   double& Y) {
  A = dot3(b[0], b[0]);
  B = dot3(b[1], b[1]);
  C = dot3(b[2], b[2]);
  E = 2.0 * dot3(b[1], b[2]);
  N = 2.0 * dot3(b[0], b[2]);
  Y = 2.0 * dot3(b[0], b[1]);
}

__device__ __forceinline__ double sgn(double x) { return x > 0.0 ? 1.0 : (x < 0.0 ? -1.0 : 0.0); }

// Krivy-Gruber on the rows of b (after LLL), the row operations applied to the integer transform T as well.  The
// steps and their tolerances are pymatgen's get_niggli_reduced_lattice.  False if it did not converge.
__device__ __noinline__ bool niggli_reduce(double (&b)[3][3], double (&T)[3][3], double e) {
  for (int it = 0; it < kNiggliIters; ++it) {
    double A, B, C, E, N, Y;
    g6(b, A, B, C, E, N, Y);
    if (A > B + e || (fabs(A - B) < e && fabs(E) > fabs(N) + e)) {          // A1: b0, b1, b2 <- -b1, -b0, -b2
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        double t = b[0][c];
        b[0][c] = -b[1][c];
        b[1][c] = -t;
        b[2][c] = -b[2][c];
        t = T[0][c];
        T[0][c] = -T[1][c];
        T[1][c] = -t;
        T[2][c] = -T[2][c];
      }
      g6(b, A, B, C, E, N, Y);
    }
    if (B > C + e || (fabs(B - C) < e && fabs(N) > fabs(Y) + e)) {          // A2: b0, b1, b2 <- -b0, -b2, -b1
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        double t = b[1][c];
        b[0][c] = -b[0][c];
        b[1][c] = -b[2][c];
        b[2][c] = -t;
        t = T[1][c];
        T[0][c] = -T[0][c];
        T[1][c] = -T[2][c];
        T[2][c] = -t;
      }
      continue;
    }
    const double l = fabs(E) < e ? 0.0 : sgn(E), m = fabs(N) < e ? 0.0 : sgn(N), n = fabs(Y) < e ? 0.0 : sgn(Y);
    double d[3];
    if (l * m * n == 1.0) {                                                 // A3
      d[0] = l == -1.0 ? -1.0 : 1.0;
      d[1] = m == -1.0 ? -1.0 : 1.0;
      d[2] = n == -1.0 ? -1.0 : 1.0;
    } else {                                                                // A4
      d[0] = l == 1.0 ? -1.0 : 1.0;
      d[1] = m == 1.0 ? -1.0 : 1.0;
      d[2] = n == 1.0 ? -1.0 : 1.0;
      if (d[0] * d[1] * d[2] == -1.0) {
        if (n == 0.0) d[2] = -1.0;
        else if (m == 0.0) d[1] = -1.0;
        else if (l == 0.0) d[0] = -1.0;
      }
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        b[r][c] *= d[r];
        T[r][c] *= d[r];
      }
    g6(b, A, B, C, E, N, Y);
    int dst = -1, src = -1;
    double s = 0.0;
    if (fabs(E) > B + e || (fabs(E - B) < e && 2.0 * N < Y - e) || (fabs(E + B) < e && Y < -e)) {
      dst = 2; src = 1; s = sgn(E);                                         // A5
    } else if (fabs(N) > A + e || (fabs(A - N) < e && 2.0 * E < Y - e) || (fabs(A + N) < e && Y < -e)) {
      dst = 2; src = 0; s = sgn(N);                                         // A6
    } else if (fabs(Y) > A + e || (fabs(A - Y) < e && 2.0 * E < N - e) || (fabs(A + Y) < e && N < -e)) {
      dst = 1; src = 0; s = sgn(Y);                                         // A7
    }
    if (dst >= 0) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        b[dst][c] -= s * b[src][c];
        T[dst][c] -= s * T[src][c];
      }
      continue;
    }
    const double S = E + N + Y + A + B;
    if (S < -e || (fabs(S) < e && e < Y + (A + N) * 2.0)) {                // A8: b2 <- b0 + b1 + b2
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        b[2][c] = b[0][c] + b[1][c] + b[2][c];
        T[2][c] = T[0][c] + T[1][c] + T[2][c];
      }
      continue;
    }
    return true;
  }
  return false;
}

// LLL then Niggli of a lattice; R = reduced rows, Tinv = inverse of the integer transform (frac' = frac @ Tinv)
__device__ __noinline__ bool reduce_cell(const double (&L)[3][3], double (&R)[3][3], double (&Tinv)[3][3]) {
  const double e = 1e-5 * cbrt(fabs(det3(L)));
  double T[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) R[r][c] = L[r][c];
  if (!lll_reduce(R, T) || !niggli_reduce(R, T, e)) return false;
  int_inverse(T, Tinv);
  return true;
}

__device__ __forceinline__ int32_t pack3(int a, int b, int c) {
  return (a + 512) | ((b + 512) << 10) | ((c + 512) << 20);
}
__device__ __forceinline__ void unpack3(int32_t w, double* n) {
  n[0] = (double)((w & 1023) - 512);
  n[1] = (double)(((w >> 10) & 1023) - 512);
  n[2] = (double)(((w >> 20) & 1023) - 512);
}

// warp argmin of (value, index), ties to the lower index
__device__ __forceinline__ void warp_argmin(double& v, int& j) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oj = __shfl_xor_sync(0xffffffffu, j, o);
    if (ov < v || (ov == v && oj < j)) {
      v = ov;
      j = oj;
    }
  }
}

struct Mapping {          // uniform across the warp
  double lll[3][3];       // LLL basis of the average lattice (rows, Cartesian)
  double lll_tol[3];
  double norm;
};

// squared distance of the nearest of the 27 images between s2 site i and s1 site j in the LLL basis (+inf when the
// pair is outside lll_frac_tol); the short vector in vec
__device__ __forceinline__ double pair_cost(const PairSmem& s, const Mapping& mp, int i, int j, double* vec) {
  double d[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    d[c] = s.lf1[j][c] - s.lf2[i][c];
    if (fabs(d[c] - rint(d[c])) > mp.lll_tol[c]) return INFINITY;
  }
  double pre[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) pre[c] = fma(d[0], mp.lll[0][c], fma(d[1], mp.lll[1][c], d[2] * mp.lll[2][c]));
  double best = INFINITY;
  int kb = 0;
  for (int k = 0; k < 27; ++k) {
    double w[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) w[c] = pre[c] + s.im[k][c];
    const double d2 = dot3(w, w);
    if (d2 < best) {
      best = d2;
      kb = k;
    }
  }
  if (vec)
#pragma unroll
    for (int c = 0; c < 3; ++c) vec[c] = pre[c] + s.im[kb][c];
  return best;
}

// Minimum-cost perfect matching of the element block [b0, b1) (rows s2 sites, columns s1 sites), shortest augmenting
// paths with the columns spread over the lanes; row_of filled.  False if no complete matching exists.
__device__ bool assign_block(PairSmem& s, const Mapping& mp, int b0, int b1, int lane) {
  const int m = b1 - b0;
  for (int j = lane; j <= m; j += 32) {
    s.u[j] = 0.0;
    s.v[j] = 0.0;
    s.p[j] = 0;
  }
  __syncwarp();
  for (int i = 1; i <= m; ++i) {
    for (int j = lane; j <= m; j += 32) {
      s.minv[j] = INFINITY;
      s.used[j] = 0;
    }
    if (lane == 0) s.p[0] = (int16_t)i;
    __syncwarp();
    int j0 = 0;
    do {
      if (lane == 0) s.used[j0] = 1;
      __syncwarp();
      const int i0 = s.p[j0];
      const double ui0 = s.u[i0];
      double delta = INFINITY;
      int j1 = 1 << 30;
      for (int j = 1 + lane; j <= m; j += 32) {
        if (s.used[j]) continue;
        const double cur = pair_cost(s, mp, b0 + i0 - 1, b0 + j - 1, nullptr) - ui0 - s.v[j];
        if (cur < s.minv[j]) {
          s.minv[j] = cur;
          s.way[j] = (int16_t)j0;
        }
        if (s.minv[j] < delta) {
          delta = s.minv[j];
          j1 = j;
        }
      }
      warp_argmin(delta, j1);
      if (delta == INFINITY) return false;
      __syncwarp();
      for (int j = lane; j <= m; j += 32) {
        if (s.used[j]) {
          s.u[s.p[j]] += delta;
          s.v[j] -= delta;
        } else {
          s.minv[j] -= delta;
        }
      }
      __syncwarp();
      j0 = j1;
    } while (s.p[j0] != 0);
    __syncwarp();          // every lane has read p[j0] before lane 0 rewrites p along the path
    if (lane == 0) {
      do {
        const int j1 = s.way[j0];
        s.p[j0] = s.p[j1];
        j0 = j1;
      } while (j0);
    }
    __syncwarp();
  }
  for (int j = 1 + lane; j <= m; j += 32) s.row_of[b0 + j - 1] = (int16_t)(b0 + s.p[j] - 1);
  __syncwarp();
  return true;
}

// first atom of the block that holds atom k of a Z-sorted crystal, and its end
__device__ __forceinline__ int block_end(const int64_t* z, int n, int b0) {
  int b1 = b0 + 1;
  while (b1 < n && z[b1] == z[b0]) ++b1;
  return b1;
}

// kFit = false: pair g is crystal g of both sets, the objective is the rms (get_rms_dist).  kFit = true: pair g is
// crystal index1[g] of set 1 (C1 crystals) against crystal index2[g] of set 2 (C2 crystals), the objective is the
// largest distance (fit), and the search stops at the first candidate below stol; rms_out is not written.
template <bool kFit>
__global__ void __launch_bounds__(32) structure_match_kernel(
    const double* __restrict__ frac1, const double* __restrict__ lattice1, const int64_t* __restrict__ z1,
    const int32_t* __restrict__ offset1, const double* __restrict__ frac2, const double* __restrict__ lattice2,
    const int64_t* __restrict__ z2, const int32_t* __restrict__ offset2, int32_t N1, int32_t N2, int32_t G,
    double stol, double ltol, double angle_tol, double* __restrict__ rms_out, double* __restrict__ max_dist_out,
    int32_t* __restrict__ num_mappings_out, int32_t* __restrict__ flags_out, const int32_t* __restrict__ index1,
    const int32_t* __restrict__ index2, int32_t C1, int32_t C2) {
  __shared__ PairSmem s;
  const int lane = threadIdx.x;
  const int g = blockIdx.x;
  if (g >= G) return;
  int x1 = g, x2 = g;                 // the crystals of the pair in set 1 and set 2
  bool bad_index = false;
  if constexpr (kFit) {
    x1 = index1[g];
    x2 = index2[g];
    bad_index = !(x1 >= 0 && x1 < C1 && x2 >= 0 && x2 < C2);
    if (bad_index) x1 = x2 = 0;
  }
  const int a0 = bad_index ? 0 : offset1[x1], a1 = bad_index ? 0 : offset1[x1 + 1];
  const int c0 = bad_index ? 0 : offset2[x2], c1 = bad_index ? 0 : offset2[x2 + 1];
  const bool bad_offsets = bad_index || !(a0 >= 0 && a1 >= a0 && a1 <= N1 && c0 >= 0 && c1 >= c0 && c1 <= N2);
  int flags = 0, num_mappings = 0;
  double best_rms = NAN, best_max = NAN;
  const int n = bad_offsets ? 0 : a1 - a0;
  const int64_t* za = z1 + a0;
  const int64_t* zb = z2 + c0;
  const double* fa = frac1 + (int64_t)a0 * 3;
  const double* fb = frac2 + (int64_t)c0 * 3;

  // ---- composition, size, finiteness, Z order ----
  if (bad_offsets) {
    flags = ARREAU_MATCH_DEGENERATE;
  } else if (c1 - c0 != n) {
    flags = ARREAU_MATCH_COMPOSITION;
  } else {
    bool differ = false, unsorted = false, finite = true;
    for (int k = lane; k < n; k += 32) {
      differ = differ || za[k] != zb[k];
      unsorted = unsorted || (k + 1 < n && (za[k] > za[k + 1] || zb[k] > zb[k + 1]));
#pragma unroll
      for (int c = 0; c < 3; ++c) finite = finite && isfinite(fa[k * 3 + c]) && isfinite(fb[k * 3 + c]);
    }
    if (__any_sync(0xffffffffu, differ)) flags = ARREAU_MATCH_COMPOSITION;
    else if (n > kMaxAtoms) flags = ARREAU_MATCH_TOO_LARGE;
    else if (n == 0 || __any_sync(0xffffffffu, unsorted) || !__all_sync(0xffffffffu, finite))
      flags = ARREAU_MATCH_DEGENERATE;
  }

  double L1[3][3], L2[3][3], T1inv[3][3], T2inv[3][3];
  if (flags == 0) {
    bool finite = true;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        L1[r][c] = lattice1[(int64_t)x1 * 9 + r * 3 + c];
        L2[r][c] = lattice2[(int64_t)x2 * 9 + r * 3 + c];
        finite = finite && isfinite(L1[r][c]) && isfinite(L2[r][c]);
      }
    if (!finite || !(fabs(det3(L1)) >= kMinVolume) || !(fabs(det3(L2)) >= kMinVolume)) {
      flags = ARREAU_MATCH_DEGENERATE;
    } else {
      double R1[3][3], R2[3][3];
      if (!reduce_cell(L1, R1, T1inv) || !reduce_cell(L2, R2, T2inv)) {
        flags = ARREAU_MATCH_DEGENERATE;
      } else {
        const double ratio = pow(fabs(det3(R2)) / fabs(det3(R1)), 1.0 / 6.0);
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            L1[r][c] = R1[r][c] * ratio;
            L2[r][c] = R2[r][c] / ratio;
          }
      }
    }
  }

  // ---- s2 in its Niggli basis; the bands of s1's lattice points ----
  double p2[6];
  int cnt[3] = {0, 0, 0};
  if (flags == 0) {
    for (int k = lane; k < n; k += 32) {
      double y[3];
      vecmat(fb + k * 3, T2inv, y);
#pragma unroll
      for (int c = 0; c < 3; ++c) s.f2[k][c] = wrap01(y[c]);
    }
    lattice_params(L2, p2);
    const double rmax = fmax(p2[0], fmax(p2[1], p2[2])) * (1.0 + ltol);
    double rinv[3];
    recip_lengths(L1, rinv);
    int K[3];
    bool too_far = false;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const double k = floor(rmax * rinv[c]);
      too_far = too_far || !(k <= kMaxSteps);
      K[c] = too_far ? 0 : (int)k;
    }
    if (too_far) {
      flags = ARREAU_MATCH_SEARCH_LIMIT;
    } else {
      const double lo = 1.0 / (1.0 + ltol), hi = 1.0 + ltol;
      const int64_t s1 = 2 * K[1] + 1, s2 = 2 * K[2] + 1, total = (int64_t)(2 * K[0] + 1) * s1 * s2;
      bool over = false;
      for (int64_t base = 0; base < total && !over; base += 32) {
        const int64_t q = base + lane;
        bool in[3] = {false, false, false};
        int32_t packed = 0;
        if (q < total) {
          const int n0 = (int)(q / (s1 * s2)) - K[0], n1 = (int)((q / s2) % s1) - K[1], n2 = (int)(q % s2) - K[2];
          const double nv[3] = {(double)n0, (double)n1, (double)n2};
          double v[3];
          vecmat(nv, L1, v);
          const double d = sqrt(dot3(v, v));
#pragma unroll
          for (int b = 0; b < 3; ++b) {
            const double r = d / p2[b];
            in[b] = r < hi && r > lo;
          }
          packed = pack3(n0, n1, n2);
        }
#pragma unroll
        for (int b = 0; b < 3; ++b) {
          const unsigned bal = __ballot_sync(0xffffffffu, in[b]);
          const int pos = cnt[b] + __popc(bal & ((1u << lane) - 1u));
          if (in[b] && pos < kBandCap) s.band[b][pos] = packed;
          cnt[b] += __popc(bal);
          over = over || cnt[b] > kBandCap;
        }
      }
      if (over) flags = ARREAU_MATCH_SEARCH_LIMIT;
    }
  }
  __syncwarp();

  if (flags == 0) {
    // angle tests between bands (x, y): alpha (b, c), beta (a, c), gamma (a, b)
    const int bx[3] = {1, 0, 0}, by[3] = {2, 2, 1};
    for (int t = 0; t < 3; ++t) {
      for (int x = 0; x < cnt[bx[t]]; ++x) {
        double nx[3], vx[3];
        unpack3(s.band[bx[t]][x], nx);
        vecmat(nx, L1, vx);
        const double dx = sqrt(dot3(vx, vx));
        for (int base = 0; base < kBandCap; base += 32) {
          const int y = base + lane;
          bool ok = false;
          if (y < cnt[by[t]]) {
            double ny[3], vy[3];
            unpack3(s.band[by[t]][y], ny);
            vecmat(ny, L1, vy);
            const double dy = sqrt(dot3(vy, vy));
            const double cosv = fmin(1.0, fmax(-1.0, dot3(vx, vy) / dx / dy));
            ok = fabs(acos(cosv) * 180.0 / M_PI - p2[3 + t]) < angle_tol;
          }
          const unsigned bal = __ballot_sync(0xffffffffu, ok);
          if (lane == 0) s.mask[t][x][base / 32] = bal;
        }
      }
    }
    // anchor: first s2 site of the rarest element (the smallest Z among ties)
    int anchor = 0, anchor_end = n, best_size = n + 1;
    for (int b0 = 0; b0 < n;) {
      const int b1 = block_end(zb, n, b0);
      if (b1 - b0 < best_size) {
        best_size = b1 - b0;
        anchor = b0;
        anchor_end = b1;
      }
      b0 = b1;
    }
    __syncwarp();
    double best = INFINITY, best_md = NAN;
    bool found = false;       // kFit: a candidate below stol was found (warp-uniform); every loop ends
    for (int ia = 0; ia < cnt[0] && !(kFit && found); ++ia) {
      for (int ib = 0; ib < cnt[1] && !(kFit && found); ++ib) {
        if (!((s.mask[2][ia][ib >> 5] >> (ib & 31)) & 1u)) continue;
        for (int w = 0; w < kBandCap / 32 && !(kFit && found); ++w) {
          unsigned bits = s.mask[0][ib][w] & s.mask[1][ia][w];
          while (bits && !(kFit && found)) {
            const int ic = w * 32 + __ffs(bits) - 1;
            bits &= bits - 1;
            if (ic >= cnt[2]) break;
            double S[3][3];
            unpack3(s.band[0][ia], S[0]);
            unpack3(s.band[1][ib], S[1]);
            unpack3(s.band[2][ic], S[2]);
            if (fabs(det3(S)) != 1.0) continue;
            ++num_mappings;
            // ---- per mapping: s1 in the mapped basis, the average lattice and its tolerances ----
            double Sinv[3][3], M[3][3], pm[6], pav[6], avg[3][3];
            int_inverse(S, Sinv);
#pragma unroll
            for (int r = 0; r < 3; ++r) vecmat(S[r], L1, M[r]);
            lattice_params(M, pm);
#pragma unroll
            for (int q = 0; q < 6; ++q) pav[q] = (pm[q] + p2[q]) / 2.0;
            lattice_from_params(pav, avg);
            Mapping mp;
            mp.norm = cbrt((double)n / fabs(det3(avg)));
            double ftol[3], rav[3], map[3][3], mapinv[3][3];
            recip_lengths(avg, rav);
#pragma unroll
            for (int c = 0; c < 3; ++c) ftol[c] = 2.0 * stol * rav[c] / mp.norm;
#pragma unroll
            for (int r = 0; r < 3; ++r)
#pragma unroll
              for (int c = 0; c < 3; ++c) mp.lll[r][c] = avg[r][c];
            lll_reduce(mp.lll, map);
            recip_lengths(mp.lll, rav);
#pragma unroll
            for (int c = 0; c < 3; ++c) mp.lll_tol[c] = 2.0 * stol * rav[c] / mp.norm;
            int_inverse(map, mapinv);
            for (int k = lane; k < n; k += 32) {
              double x[3], y[3];
              vecmat(fa + k * 3, T1inv, x);
#pragma unroll
              for (int c = 0; c < 3; ++c) x[c] = wrap01(x[c]);
              vecmat(x, Sinv, y);
#pragma unroll
              for (int c = 0; c < 3; ++c) s.fc1[k][c] = wrap01(y[c]);
              vecmat(s.fc1[k], mapinv, y);
#pragma unroll
              for (int c = 0; c < 3; ++c) s.lf1[k][c] = wrap01(y[c]);
            }
            if (lane < 27) {
              const double kv[3] = {(double)(lane / 9 - 1), (double)((lane / 3) % 3 - 1), (double)(lane % 3 - 1)};
              vecmat(kv, mp.lll, s.im[lane]);
            }
            __syncwarp();
            // ---- translations ----
            for (int jt = anchor; jt < anchor_end; ++jt) {
              __syncwarp();        // the previous translation's reads of lf2 are done
              double t[3];
#pragma unroll
              for (int c = 0; c < 3; ++c) t[c] = s.fc1[jt][c] - s.f2[anchor][c];
              bool ok = true;
              int b0 = 0, b1 = 0;
              for (int base = 0; base < n && ok; base += 32) {
                const int i = base + lane;
                bool found = true;
                if (i < n) {
                  if (i >= b1 || i < b0) {      // the element block of site i
                    b0 = i;
                    while (b0 > 0 && zb[b0 - 1] == zb[i]) --b0;
                    b1 = block_end(zb, n, i);
                  }
                  found = false;
                  for (int j = b0; j < b1 && !found; ++j) {
                    bool in = true;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                      const double d = s.f2[i][c] + t[c] - s.fc1[j][c];
                      in = in && fabs(d - rint(d)) <= ftol[c];
                    }
                    found = in;
                  }
                }
                ok = __all_sync(0xffffffffu, found);
              }
              if (!ok) continue;
              for (int k = lane; k < n; k += 32) {
                double x[3], y[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) x[c] = s.f2[k][c] + t[c];
                vecmat(x, mapinv, y);
#pragma unroll
                for (int c = 0; c < 3; ++c) s.lf2[k][c] = wrap01(y[c]);
              }
              __syncwarp();
              bool feasible = true;
              for (int e0 = 0; e0 < n && feasible;) {
                const int e1 = block_end(zb, n, e0);
                feasible = assign_block(s, mp, e0, e1, lane);
                e0 = e1;
              }
              __syncwarp();
              if (!feasible) continue;
              // distances from the matched short vectors less their mean
              double sum[3] = {0.0, 0.0, 0.0};
              for (int j = lane; j < n; j += 32) {
                double vec[3];
                pair_cost(s, mp, s.row_of[j], j, vec);
#pragma unroll
                for (int c = 0; c < 3; ++c) sum[c] += vec[c];
              }
              double mean[3];
#pragma unroll
              for (int c = 0; c < 3; ++c) mean[c] = warp_sum(sum[c]) / (double)n;
              double sq = 0.0, mx = 0.0;
              for (int j = lane; j < n; j += 32) {
                double vec[3];
                pair_cost(s, mp, s.row_of[j], j, vec);
#pragma unroll
                for (int c = 0; c < 3; ++c) vec[c] -= mean[c];
                const double dist = sqrt(dot3(vec, vec)) * mp.norm;
                sq = fma(dist, dist, sq);
                mx = fmax(mx, dist);
              }
              if constexpr (kFit) {
                mx = warp_max(mx);
                if (mx < best) best = mx;
                if (mx < stol) {
                  found = true;
                  break;
                }
              } else {
                const double rms = sqrt(warp_sum(sq)) / sqrt((double)n);
                mx = warp_max(mx);
                if (rms < best) {
                  best = rms;
                  best_md = mx;
                }
              }
            }
            __syncwarp();
          }
        }
      }
    }
    if (best < INFINITY) {
      best_rms = best;
      best_max = kFit ? best : best_md;
      if (best < stol) flags = ARREAU_MATCH_MATCHED;
    }
  }

  if (lane == 0) {
    if constexpr (!kFit) rms_out[g] = best_rms;
    max_dist_out[g] = best_max;
    num_mappings_out[g] = num_mappings;
    flags_out[g] = flags;
  }
}

}  // namespace

extern "C" int arreau_structure_match(const double* frac1, const double* lattice1, const int64_t* z1,
                                      const int32_t* offset1, const double* frac2, const double* lattice2,
                                      const int64_t* z2, const int32_t* offset2, int32_t num_atoms1,
                                      int32_t num_atoms2, int32_t num_pairs, double stol, double ltol,
                                      double angle_tol, double* rms, double* max_dist, int32_t* num_mappings,
                                      int32_t* flags, void* stream) {
  if (num_pairs == 0) return ARREAU_OK;
  if (!lattice1 || !offset1 || !lattice2 || !offset2 || !rms || !max_dist || !num_mappings || !flags)
    return ARREAU_ERR_NULL;
  if ((num_atoms1 > 0 && (!frac1 || !z1)) || (num_atoms2 > 0 && (!frac2 || !z2))) return ARREAU_ERR_NULL;
  if (num_pairs < 0 || num_atoms1 < 0 || num_atoms2 < 0 || !(stol > 0.0) || !(ltol > 0.0) || !(angle_tol > 0.0) ||
      !isfinite(stol) || !isfinite(ltol) || !isfinite(angle_tol))
    return ARREAU_ERR_BAD_SHAPE;
  structure_match_kernel<false><<<(unsigned)num_pairs, 32, 0, (cudaStream_t)stream>>>(
      frac1, lattice1, z1, offset1, frac2, lattice2, z2, offset2, num_atoms1, num_atoms2, num_pairs, stol, ltol,
      angle_tol, rms, max_dist, num_mappings, flags, nullptr, nullptr, num_pairs, num_pairs);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_structure_fit_pairs(const double* frac1, const double* lattice1, const int64_t* z1,
                                          const int32_t* offset1, int32_t num_atoms1, int32_t num_crystals1,
                                          const double* frac2, const double* lattice2, const int64_t* z2,
                                          const int32_t* offset2, int32_t num_atoms2, int32_t num_crystals2,
                                          const int32_t* index1, const int32_t* index2, int32_t num_pairs,
                                          double stol, double ltol, double angle_tol, double* max_dist,
                                          int32_t* num_mappings, int32_t* flags, void* stream) {
  if (num_pairs == 0) return ARREAU_OK;
  if (!lattice1 || !offset1 || !lattice2 || !offset2 || !index1 || !index2 || !max_dist || !num_mappings || !flags)
    return ARREAU_ERR_NULL;
  if ((num_atoms1 > 0 && (!frac1 || !z1)) || (num_atoms2 > 0 && (!frac2 || !z2))) return ARREAU_ERR_NULL;
  if (num_pairs < 0 || num_atoms1 < 0 || num_atoms2 < 0 || num_crystals1 < 0 || num_crystals2 < 0 || !(stol > 0.0) ||
      !(ltol > 0.0) || !(angle_tol > 0.0) || !isfinite(stol) || !isfinite(ltol) || !isfinite(angle_tol))
    return ARREAU_ERR_BAD_SHAPE;
  structure_match_kernel<true><<<(unsigned)num_pairs, 32, 0, (cudaStream_t)stream>>>(
      frac1, lattice1, z1, offset1, frac2, lattice2, z2, offset2, num_atoms1, num_atoms2, num_pairs, stol, ltol,
      angle_tol, nullptr, max_dist, num_mappings, flags, index1, index2, num_crystals1, num_crystals2);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}
