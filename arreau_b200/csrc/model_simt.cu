// K2-K7 of the Ponita fiber-bundle forward in fp32 (sm_100a, FFMA2 SIMT path).
//
// This is the fp32-grade path (parity within 1e-4 of the fp64 reference).  The dense contractions
// run as shared-memory tiled SIMT GEMMs on packed FFMA2; the tcgen05 fp16 variants of the two
// GEMM-shaped kernels live in model_tc.cu and share every other kernel in this file.
//
//   node_embed_kernel          K2   position_orientation_graph.py:84-86 + ponita.py:98
//   fiber_kernel_kernel        K3'  geometry/invariants.py:23, ponita.py:66,95, conv.py:113
//   edge_kernels_simt_kernel   K3+K4a  invariants -> monomials -> basis MLP -> window -> 5 kernel projections
//   message_fiber_norm_kernel  K4b+K5 + LayerNorm   conv.py:115,126-133, convnext.py:25
//   convnext_mlp_simt_kernel   K6   convnext.py:26-32
//   readout_*_kernel           K7   ponita.py:105-117,152, to_from_sphere.py:10-14
#include <cstdlib>
#include <cuda_fp16.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace {

// ------------------------------------------------------------------------------------------------
// shared SIMT GEMM pass:  acc[128 x 128] += A^T(smem [K][kPitch]) * B(global [K][ldb], 128 columns)
// 256 threads, thread (ty, tx) owns rows {ty*4..+3, 64+ty*4..+3} x cols {tx*4..+3, 64+tx*4..+3}.
// B is streamed through a cp.async double buffer in chunks of kKC rows.
// ------------------------------------------------------------------------------------------------
constexpr int kTM = 128;
constexpr int kPitch = 132;
constexpr int kKC = 16;
constexpr int kNT = 128;
constexpr int kGemmThreads = 256;

__device__ __forceinline__ void zero_acc(float2 (&acc)[8][4]) {
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.f, 0.f);
}

__device__ __forceinline__ int acc_row(int ty, int i) { return (i < 4) ? (ty * 4 + i) : (64 + ty * 4 + i - 4); }
__device__ __forceinline__ int acc_col(int tx, int j2) {  // j2 in 0..7
  return (j2 < 4) ? (tx * 4 + j2) : (64 + tx * 4 + j2 - 4);
}

template <int K>
__device__ __forceinline__ void gemm_pass(float2 (&acc)[8][4], const float* __restrict__ As,
                                          const float* __restrict__ Bg, int ldb, float* __restrict__ Bs, int tid) {
  static_assert(K % kKC == 0, "K must be a multiple of the chunk");
  const int ty = tid >> 4, tx = tid & 15;
  auto load_chunk = [&](int chunk, int buf) {
#pragma unroll
    for (int v = tid; v < kKC * kNT / 4; v += kGemmThreads) {
      const int r = v >> 5, c4 = v & 31;
      cp_async16(Bs + buf * kKC * kNT + r * kNT + c4 * 4, Bg + (size_t)(chunk * kKC + r) * ldb + c4 * 4);
    }
    cp_async_commit();
  };
  load_chunk(0, 0);
  constexpr int kChunks = K / kKC;
  for (int ch = 0; ch < kChunks; ++ch) {
    if (ch + 1 < kChunks) {
      load_chunk(ch + 1, (ch + 1) & 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* b = Bs + (ch & 1) * kKC * kNT;
    const float* a = As + ch * kKC * kPitch;
#pragma unroll
    for (int k = 0; k < kKC; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(a + k * kPitch + ty * 4);
      const float4 a1 = *reinterpret_cast<const float4*>(a + k * kPitch + 64 + ty * 4);
      const float4 b0 = *reinterpret_cast<const float4*>(b + k * kNT + tx * 4);
      const float4 b1 = *reinterpret_cast<const float4*>(b + k * kNT + 64 + tx * 4);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float2 bv[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y),
                            make_float2(b1.z, b1.w)};
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 aa = make_float2(av[i], av[i]);
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = __ffma2_rn(aa, bv[j], acc[i][j]);
      }
    }
    __syncthreads();
  }
}

// acc element (i, j2) with j2 in 0..7
__device__ __forceinline__ float acc_get(const float2 (&acc)[8][4], int i, int j2) {
  return (j2 & 1) ? acc[i][j2 >> 1].y : acc[i][j2 >> 1].x;
}

// ------------------------------------------------------------------------------------------------
// K2  node embedding
// ------------------------------------------------------------------------------------------------
constexpr int kEmbedNodes = 8;
constexpr int kMaxVec = 8;

// thread = (atom a of the CTA's 8, 4 channels): s = sum_f x[b,f] W[f, 4 cg..] once per atom, then the 16 orientations
// only add the vector part (linearity) and store 16 bytes.  `types` (optional): the first Z features are a one-hot of
// types[b] (diffusion_loss.py:140-150) -> one row lookup instead of Z multiply-adds with zeros.
// kV > 0: the number of vector channels at compile time (4 in the diffusion model: no predicated-off slots)
template <int kV>
__global__ void __launch_bounds__(kEmbedNodes * 32)
node_embed_kernel(const float* __restrict__ x, const float* __restrict__ vec, const float* __restrict__ w_t,
                  const float* __restrict__ ori, const int64_t* __restrict__ types, int Z, int N, int F, int V_rt,
                  float* __restrict__ h, float* __restrict__ pool, const float* __restrict__ pool_wz, int pool_z) {
  const int V = kV > 0 ? kV : V_rt;
  constexpr int kVecSlots = kV > 0 ? kV : kMaxVec;
  extern __shared__ float sm[];
  float* xs = sm;                                   // [kEmbedNodes][F]
  float* dots = sm + kEmbedNodes * F;               // [kEmbedNodes][V][kO]
  const int tid = threadIdx.x, a = tid >> 5, lane = tid & 31;
  const int b0 = blockIdx.x * kEmbedNodes;
  const int nb = min(kEmbedNodes, N - b0);
  for (int idx = tid; idx < nb * F; idx += kEmbedNodes * 32) xs[idx] = x[(size_t)b0 * F + idx];
  for (int idx = tid; idx < nb * V * kO; idx += kEmbedNodes * 32) {
    const int o = idx % kO, v = (idx / kO) % V, b = idx / (kO * V);
    const float* p = vec + ((size_t)(b0 + b) * V + v) * 3;
    dots[idx] = p[0] * ori[3 * o] + p[1] * ori[3 * o + 1] + p[2] * ori[3 * o + 2];   // to_from_sphere.py:7-8
  }
  __syncthreads();
  // pooled read-out features by linearity: sum_o w_o h[b,o,:] = (sum_o w_o) s + sum_v (sum_o w_o dots[b,v,o]) W_v for the
  // four weightings w = 1, ori[:,0..2]; the orientation sums of the dots are formed once per atom here
  float* dred = dots + kEmbedNodes * V * kO;        // [kEmbedNodes][V][4], then osum[4] = sum_o (1, ori[o][0..2])
  if (pool) {
    for (int idx = tid; idx < nb * V * 4 + 4; idx += kEmbedNodes * 32) {
      const int q = idx & 3, bv = idx >> 2;          // bv = b * V + v, or nb * V for the weight sums themselves
      float acc = 0.f;
      for (int o = 0; o < kO; ++o) {
        const float wgt = q == 0 ? 1.0f : ori[3 * o + q - 1];
        acc += wgt * (bv < nb * V ? dots[bv * kO + o] : 1.0f);
      }
      dred[idx] = acc;
    }
    __syncthreads();
  }
  float4 pq[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) pq[q] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (a < nb) {
  const float* xr = xs + a * F;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  int f0 = 0;
  if (types) {
    s = __ldg(reinterpret_cast<const float4*>(w_t + (size_t)types[b0 + a] * kC + lane * 4));
    f0 = Z;
  }
#pragma unroll 16
  for (int f = f0; f < F; ++f) {
    const float4 w = __ldg(reinterpret_cast<const float4*>(w_t + (size_t)f * kC + lane * 4));
    const float xv = xr[f];
    s.x = fmaf(xv, w.x, s.x); s.y = fmaf(xv, w.y, s.y); s.z = fmaf(xv, w.z, s.z); s.w = fmaf(xv, w.w, s.w);
  }
  float4 wv[kVecSlots];
#pragma unroll
  for (int v = 0; v < kVecSlots; ++v)
    wv[v] = v < V ? __ldg(reinterpret_cast<const float4*>(w_t + (size_t)(F + v) * kC + lane * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
  float* hp = h + (size_t)(b0 + a) * kO * kC + lane * 4;
  // optional orientation-pooled copy for the pooled read-out (part 0 = mean_o h, part 1+d = (1/O) sum_o ori[o][d] h)
#pragma unroll 4
  for (int o = 0; o < kO; ++o) {
    float4 r = s;
#pragma unroll
    for (int v = 0; v < kVecSlots; ++v)
      if (v < V) {
        const float dv = dots[(a * V + v) * kO + o];
        r.x = fmaf(dv, wv[v].x, r.x); r.y = fmaf(dv, wv[v].y, r.y); r.z = fmaf(dv, wv[v].z, r.z); r.w = fmaf(dv, wv[v].w, r.w);
      }
    *reinterpret_cast<float4*>(hp + o * kC) = r;
  }
  if (pool) {
    const float* osum = dred + nb * V * 4;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float ws = osum[q];
      float4 acc = make_float4(ws * s.x, ws * s.y, ws * s.z, ws * s.w);
#pragma unroll
      for (int v = 0; v < kVecSlots; ++v)
        if (v < V) {
          const float dv = dred[(a * V + v) * 4 + q];
          acc.x = fmaf(dv, wv[v].x, acc.x); acc.y = fmaf(dv, wv[v].y, acc.y);
          acc.z = fmaf(dv, wv[v].z, acc.z); acc.w = fmaf(dv, wv[v].w, acc.w);
        }
      pq[q] = acc;
    }
  }
  }
  if (pool) {
    // pool entry (include/arreau_b200.h): [group of 16 atoms][C][16 atoms] of mean_o h, then per atom the 3 x 2 partial
    // contractions of the vector-pooled parts with the score row of the read-out.  The CTA's 8 atoms are one half of a
    // group; transpose [atom][c] -> [c][atom] through shared memory (re-using xs / dots)
    constexpr float inv = 1.0f / kO;
    const int groups = (N + 15) / 16;
    if (a < nb) {
      float sd[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        const float* wz = pool_wz + (size_t)(lane * 4) * (pool_z + 6) + pool_z;     // V_0[c][Z], c = 4 lane + i
        float v = pq[1 + d].x * wz[0] + pq[1 + d].y * wz[pool_z + 6] + pq[1 + d].z * wz[2 * (pool_z + 6)] +
                  pq[1 + d].w * wz[3 * (pool_z + 6)];
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
        sd[d] = v * inv;
      }
      if (lane == 0) {
        float4* sp = reinterpret_cast<float4*>(pool + (size_t)groups * kC * 16 + (size_t)(b0 + a) * 8);
        sp[0] = make_float4(sd[0], 0.f, sd[1], 0.f);                                // [2 d + half]: this kernel fills half 0
        sp[1] = make_float4(sd[2], 0.f, 0.f, 0.f);
      }
    }
    __syncthreads();
    float* tp = sm;                                            // [8 atoms][kC]
    *reinterpret_cast<float4*>(tp + a * kC + lane * 4) = make_float4(pq[0].x * inv, pq[0].y * inv, pq[0].z * inv, pq[0].w * inv);
    __syncthreads();
    float* pg = pool + (size_t)(blockIdx.x >> 1) * kC * 16 + (size_t)(blockIdx.x & 1) * 8;
    for (int pc = tid; pc < kC; pc += kEmbedNodes * 32) {
      float v[8];
#pragma unroll
      for (int aa = 0; aa < 8; ++aa) v[aa] = tp[aa * kC + pc];
      float4* po = reinterpret_cast<float4*>(pg + (size_t)pc * 16);
      po[0] = make_float4(v[0], v[1], v[2], v[3]);
      po[1] = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K3'  fiber kernels (input independent; evaluated in fp64, stored fp32)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ double gelu_erf_d(double x) { return 0.5 * x * (1.0 + erf(x * 0.70710678118654752440)); }

__global__ void __launch_bounds__(kD)
fiber_kernel_kernel(const float* __restrict__ ori, const float* __restrict__ w1, const float* __restrict__ b1,
                    const float* __restrict__ w2, const float* __restrict__ b2, const float* __restrict__ wf,
                    float* __restrict__ fk) {
  __shared__ double h1[kC];
  __shared__ double fkb[kD];
  const int o = blockIdx.x / kO, p = blockIdx.x % kO, t = threadIdx.x;
  const double fa = (double)ori[3 * o] * ori[3 * p] + (double)ori[3 * o + 1] * ori[3 * p + 1] +
                    (double)ori[3 * o + 2] * ori[3 * p + 2];
  if (t < kC) h1[t] = gelu_erf_d(w1[3 * t] * fa + w1[3 * t + 1] * (fa * fa) + w1[3 * t + 2] * (fa * fa * fa) + b1[t]);
  __syncthreads();
  // a warp per output, lanes over the reduced index (coalesced weight rows, shuffle tree): one thread per output walking
  // a 1 KB-strided row of 256 fp64 products took 213 us per call, once per training step
  const int warp = t >> 5, lane = t & 31;
  auto warp_sum = [](double s) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    return s;
  };
  // four outputs per pass: their weight rows are loaded together (one memory round trip per pass, not per output)
  for (int d0 = warp * 4; d0 < kD; d0 += kD / 8) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float* w = w2 + (size_t)(d0 + u) * kC;
#pragma unroll
      for (int c = lane; c < kC; c += 32) s[u] += (double)w[c] * h1[c];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double t4 = warp_sum(s[u]);
      if (lane == 0) fkb[d0 + u] = t4 + (double)b2[d0 + u];
    }
  }
  __syncthreads();
  fkb[t] = gelu_erf_d(fkb[t]);           // one fp64 erf per thread (kD threads), not 32 in a row on lane 0 of each warp
  __syncthreads();
  for (int i0 = warp * 4; i0 < kL * kC; i0 += kD / 8) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float* w = wf + (size_t)(i0 + u) * kD;         // row (l, c) = i0 + u of wf[L][C][D]
#pragma unroll
      for (int d = lane; d < kD; d += 32) s[u] += (double)w[d] * fkb[d];
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double t4 = warp_sum(s[u]);
      const int l = (i0 + u) / kC, c = (i0 + u) % kC;
      if (lane == 0) fk[(((size_t)l * kO + o) * kO + p) * kC + c] = (float)t4;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K3 + K4a  edge pipeline (fp32 SIMT)
// ------------------------------------------------------------------------------------------------
constexpr int kEdgesPerTile = kTM / kO;   // 8
constexpr size_t kEdgeSmemFloats = (size_t)kD * kPitch + (size_t)kC * kPitch + 2 * kKC * kNT;

__global__ void __launch_bounds__(kGemmThreads, 1)
edge_kernels_simt_kernel(const double* __restrict__ dir, const double* __restrict__ dist,
                         const double* __restrict__ lattice, const int32_t* __restrict__ crystal_of_atom,
                         const int32_t* __restrict__ src, const int32_t* __restrict__ num_edges_ptr,
                         long long edge_capacity, const float* __restrict__ ori, const float* __restrict__ w1m_t,
                         const float* __restrict__ w2_t, const float* __restrict__ b2,
                         const float* __restrict__ wk_t, double radius, float* __restrict__ kernels) {
  extern __shared__ __align__(16) float smem[];
  float* Xs = smem;                      // [kD][kPitch]: monomials (rows 0..95), later the kernel basis
  float* Ys = Xs + kD * kPitch;          // [kC][kPitch]: hidden layer of the basis MLP
  float* Bs = Ys + kC * kPitch;          // [2][kKC][kNT]
  __shared__ float s_win[kEdgesPerTile];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  long long E = *num_edges_ptr;
  if (E > edge_capacity) E = edge_capacity;
  const long long tiles = (E + kEdgesPerTile - 1) / kEdgesPerTile;
  float2 acc[8][4];
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    // ---- invariants -> 83 monomials + constant 1 (bias row) + zero padding to 96 ----
    if (tid < kTM) {
      const int row = tid, o = row & (kO - 1);
      const long long e = tile * kEdgesPerTile + (row >> 4);
      float attr[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      float one = 0.f;
      if (e < E) {
        const int g = crystal_of_atom[src[e]];
        edge_invariants(dir + 3 * e, dist[e], lattice + 9 * (size_t)g, ori + 3 * o, attr);
        one = 1.f;
        if (o == 0) s_win[row >> 4] = cutoff_window(dist[e], radius);
      } else if (o == 0) {
        s_win[row >> 4] = 0.f;
      }
      monomials83(attr, Xs + row, kPitch);
      Xs[kMono * kPitch + row] = one;
#pragma unroll
      for (int k = kMono + 1; k < kMonoPad; ++k) Xs[k * kPitch + row] = 0.f;
    }
    __syncthreads();
    // ---- hidden = GELU(W1m . monomials)   (bias folded into the constant row) ----
    zero_acc(acc);
    gemm_pass<kMonoPad>(acc, Xs, w1m_t, kC, Bs, tid);
#pragma unroll
    for (int j2 = 0; j2 < 8; ++j2) {
      const int n = acc_col(tx, j2);
      float4 lo = make_float4(gelu_erf(acc_get(acc, 0, j2)), gelu_erf(acc_get(acc, 1, j2)),
                              gelu_erf(acc_get(acc, 2, j2)), gelu_erf(acc_get(acc, 3, j2)));
      float4 hi = make_float4(gelu_erf(acc_get(acc, 4, j2)), gelu_erf(acc_get(acc, 5, j2)),
                              gelu_erf(acc_get(acc, 6, j2)), gelu_erf(acc_get(acc, 7, j2)));
      *reinterpret_cast<float4*>(Ys + n * kPitch + ty * 4) = lo;
      *reinterpret_cast<float4*>(Ys + n * kPitch + 64 + ty * 4) = hi;
    }
    // ---- kernel basis = GELU(W2 . hidden + b2) * window ----
    for (int p = 0; p < kD / kNT; ++p) {
      zero_acc(acc);
      gemm_pass<kC>(acc, Ys, w2_t + p * kNT, kD, Bs, tid);
      float wl[4], wh[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        wl[i] = s_win[(ty * 4 + i) >> 4];
        wh[i] = s_win[(64 + ty * 4 + i) >> 4];
      }
#pragma unroll
      for (int j2 = 0; j2 < 8; ++j2) {
        const int n = p * kNT + acc_col(tx, j2);
        const float bb = b2[n];
        float4 lo = make_float4(gelu_erf(acc_get(acc, 0, j2) + bb) * wl[0], gelu_erf(acc_get(acc, 1, j2) + bb) * wl[1],
                                gelu_erf(acc_get(acc, 2, j2) + bb) * wl[2], gelu_erf(acc_get(acc, 3, j2) + bb) * wl[3]);
        float4 hi = make_float4(gelu_erf(acc_get(acc, 4, j2) + bb) * wh[0], gelu_erf(acc_get(acc, 5, j2) + bb) * wh[1],
                                gelu_erf(acc_get(acc, 6, j2) + bb) * wh[2], gelu_erf(acc_get(acc, 7, j2) + bb) * wh[3]);
        *reinterpret_cast<float4*>(Xs + n * kPitch + ty * 4) = lo;
        *reinterpret_cast<float4*>(Xs + n * kPitch + 64 + ty * 4) = hi;
      }
    }
    // ---- per-layer spatial kernels = Wk_l . kernel basis  -> kernels[l][e][o][c] ----
    for (int l = 0; l < kL; ++l) {
      zero_acc(acc);
      gemm_pass<kD>(acc, Xs, wk_t + l * kNT, kL * kC, Bs, tid);
      float* out = kernels + (size_t)l * edge_capacity * kO * kC + (size_t)tile * kTM * kC;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int row = acc_row(ty, i);
        if (tile * kEdgesPerTile + (row >> 4) < E) {
          *reinterpret_cast<float4*>(out + (size_t)row * kC + tx * 4) =
              make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
          *reinterpret_cast<float4*>(out + (size_t)row * kC + 64 + tx * 4) =
              make_float4(acc[i][2].x, acc[i][2].y, acc[i][3].x, acc[i][3].y);
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// K4b + K5 + LayerNorm: receiver-sorted CSR reduction, fiber conv, norm.  Deterministic.
// 128 threads: warp og owns orientations og*4..+3, lane cg owns channels cg*4..+3.
// ------------------------------------------------------------------------------------------------

// Channels 4*cg .. +3 of kernel row (e, o).  fp32 kernels are plain [e][o][c]; fp16 kernels (tcgen05 path) keep
// the 16-byte chunk k of a row at chunk position k ^ o (so the producing kernel can stage and bulk-store its
// tiles without shared-memory bank conflicts, csrc/model_tc.cu); a warp still reads whole 256-byte rows.
__device__ __forceinline__ float4 load_kernel4(const float* row, int cg, int /*o*/) {
  return *reinterpret_cast<const float4*>(row + cg * 4);
}
__device__ __forceinline__ float4 load_kernel4(const __half* row, int cg, int o) {
  const __half* p = row + ((((cg >> 1) ^ (o & 15)) << 3) | ((cg & 1) << 2));
  const uint2 raw = *reinterpret_cast<const uint2*>(p);
  const __half2 a = *reinterpret_cast<const __half2*>(&raw.x);
  const __half2 b = *reinterpret_cast<const __half2*>(&raw.y);
  const float2 fa = __half22float2(a), fb = __half22float2(b);
  return make_float4(fa.x, fa.y, fb.x, fb.y);
}

// K4b  message_gather_kernel: one warp per (receiver, orientation), lane = 4 channels.
//        x1[i][o][c] = sum over the receiver's edges (fixed CSR order -> deterministic, no atomics) of
//        kernel[e][o][c] * h[src_e][o][c]; 8 edges (16 independent 8/16-byte loads per lane) in flight.
// K5   fiber_norm_kernel: persistent CTAs of 16 warps; thread (warp p, lane cg) keeps its 16 fiber-kernel values
//        fk[.][p][4cg..] in registers for the whole kernel and streams x1 rows (coalesced 512-byte rows):
//        x2[i][p][c] = (1/O) sum_o x1[i][o][c] fk[o][p][c] + bias[c], then LayerNorm over c as a warp reduction.
constexpr int kGatherWarps = 8;

template <typename KT, typename XT>
__global__ void __launch_bounds__(kGatherWarps * 32)
message_gather_kernel(const KT* __restrict__ kern, const float* __restrict__ h, const int32_t* __restrict__ row_ptr,
                      const int32_t* __restrict__ src, long long rows, XT* __restrict__ x1) {
  const long long r = (long long)blockIdx.x * kGatherWarps + (threadIdx.x >> 5);   // row = node * kO + o
  if (r >= rows) return;
  const int cg = threadIdx.x & 31;
  const int node = (int)(r >> 4), o = (int)(r & (kO - 1));
  const int e0 = row_ptr[node], e1 = row_ptr[node + 1];
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  int e = e0;
  for (; e + 8 <= e1; e += 8) {
    int sidx[8];
    float4 kv[8], hv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) sidx[u] = __ldg(src + e + u);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      kv[u] = load_kernel4(kern + ((size_t)(e + u) * kO + o) * kC, cg, o);
      hv[u] = *reinterpret_cast<const float4*>(h + ((size_t)sidx[u] * kO + o) * kC + cg * 4);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a.x = fmaf(kv[u].x, hv[u].x, a.x);
      a.y = fmaf(kv[u].y, hv[u].y, a.y);
      a.z = fmaf(kv[u].z, hv[u].z, a.z);
      a.w = fmaf(kv[u].w, hv[u].w, a.w);
    }
  }
  for (; e < e1; ++e) {
    const float4 kv = load_kernel4(kern + ((size_t)e * kO + o) * kC, cg, o);
    const float4 hv = *reinterpret_cast<const float4*>(h + ((size_t)__ldg(src + e) * kO + o) * kC + cg * 4);
    a.x = fmaf(kv.x, hv.x, a.x);
    a.y = fmaf(kv.y, hv.y, a.y);
    a.z = fmaf(kv.z, hv.z, a.z);
    a.w = fmaf(kv.w, hv.w, a.w);
  }
  if constexpr (sizeof(XT) == 4) {
    *reinterpret_cast<float4*>(x1 + (size_t)r * kC + cg * 4) = a;
  } else {   // fp16 path: the message sums feed a LayerNorm whose output is rounded to fp16 anyway
    __half2 p0 = __floats2half2_rn(a.x, a.y), p1 = __floats2half2_rn(a.z, a.w);
    uint2 raw;
    raw.x = *reinterpret_cast<unsigned*>(&p0);
    raw.y = *reinterpret_cast<unsigned*>(&p1);
    *reinterpret_cast<uint2*>(x1 + (size_t)r * kC + cg * 4) = raw;
  }
}

// ---- fp16 tensor path: transposed message sums + tensor-core fiber conv ----------------------------------------
// K4b (fp16 path)  message_gather_t_kernel: one CTA of 16 warps per receiver atom (warp = orientation, lane = 4
//   channels); the 16 x 128 message sums are transposed through shared memory and written as x1t[atom][c][o] fp16
//   (the 16 orientations of a channel are 32 contiguous bytes), the A-operand layout of the fiber conv below.
constexpr int kGatherTThreads = kO * 32;

__global__ void __launch_bounds__(kGatherTThreads)
message_gather_t_kernel(const __half* __restrict__ kern, const float* __restrict__ h, const int32_t* __restrict__ row_ptr,
                        const int32_t* __restrict__ src, int N, __half* __restrict__ x1t) {
  __shared__ __align__(16) __half tile[kO][kC + 8];       // +8 halfs: conflict-free column reads
  const int node = blockIdx.x, o = threadIdx.x >> 5, cg = threadIdx.x & 31;
  const int e0 = row_ptr[node], e1 = row_ptr[node + 1];
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  int e = e0;
  for (; e + 8 <= e1; e += 8) {
    int sidx[8];
    float4 kv[8], hv[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) sidx[u] = __ldg(src + e + u);
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      kv[u] = load_kernel4(kern + ((size_t)(e + u) * kO + o) * kC, cg, o);
      hv[u] = *reinterpret_cast<const float4*>(h + ((size_t)sidx[u] * kO + o) * kC + cg * 4);
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a.x = fmaf(kv[u].x, hv[u].x, a.x);
      a.y = fmaf(kv[u].y, hv[u].y, a.y);
      a.z = fmaf(kv[u].z, hv[u].z, a.z);
      a.w = fmaf(kv[u].w, hv[u].w, a.w);
    }
  }
  for (; e < e1; ++e) {
    const float4 kv = load_kernel4(kern + ((size_t)e * kO + o) * kC, cg, o);
    const float4 hv = *reinterpret_cast<const float4*>(h + ((size_t)__ldg(src + e) * kO + o) * kC + cg * 4);
    a.x = fmaf(kv.x, hv.x, a.x);
    a.y = fmaf(kv.y, hv.y, a.y);
    a.z = fmaf(kv.z, hv.z, a.z);
    a.w = fmaf(kv.w, hv.w, a.w);
  }
  {
    const __half2 p0 = __floats2half2_rn(a.x, a.y), p1 = __floats2half2_rn(a.z, a.w);
    uint2 raw;
    raw.x = *reinterpret_cast<const unsigned*>(&p0);
    raw.y = *reinterpret_cast<const unsigned*>(&p1);
    *reinterpret_cast<uint2*>(&tile[o][cg * 4]) = raw;
  }
  __syncthreads();
  {
    // thread -> (channel c, orientations 4 oq .. +3): 8 bytes, the CTA writes the atom's 4 KB contiguously
    const int c = threadIdx.x >> 2, oq = (threadIdx.x & 3) * 4;
    const __half2 p0 = __halves2half2(tile[oq][c], tile[oq + 1][c]), p1 = __halves2half2(tile[oq + 2][c], tile[oq + 3][c]);
    uint2 raw;
    raw.x = *reinterpret_cast<const unsigned*>(&p0);
    raw.y = *reinterpret_cast<const unsigned*>(&p1);
    *reinterpret_cast<uint2*>(x1t + ((size_t)node * kC + c) * kO + oq) = raw;
  }
}

// K5 (fp16 path)  fiber_norm_mma_kernel.  For a fixed channel the fiber conv is a 16 x 16 matrix product over the
//   orientations, x2[atom][p] = sum_o x1[atom][o] fk[o][p]: one warp takes 16 atoms and runs it as two
//   mma.sync.m16n8k16 (fp16 operands, fp32 accumulation) per channel, 5x fewer instructions than the SIMT form
//   (tcgen05 has no shape for a per-channel 16 x 16 x 16 product).  Every (atom, p) pair lives in exactly one lane, so
//   the LayerNorm statistics over the 128 channels need no shuffles: pass 1 accumulates sum and sum of squares,
//   pass 2 recomputes the (cheap) products, normalises and emits 8 channels = one 16-byte chunk of the ConvNext
//   kernel's UMMA operand image at a time.
//   fk_frag[c][lane] (uint4): the B fragments of channel c for the two n-tiles, with the 1/O of conv.py:115 folded in.
constexpr int kFiberMmaWarps = 8;    // warp w owns channels 16 w .. 16 w + 15 (16 warps measured slower: the statistics exchange grows)

__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1), "f"(0.f));
}

__global__ void fiber_frag_kernel(const float* __restrict__ fk, uint4* __restrict__ frag) {
  // grid = L * C blocks of 32 threads; fk[l][o][p][c]
  const int l = blockIdx.x / kC, c = blockIdx.x % kC, lane = threadIdx.x, g = lane >> 2, t = lane & 3;
  const float* f = fk + (size_t)l * kO * kO * kC + c;
  auto at = [&](int o, int p) { return f[((size_t)o * kO + p) * kC] * (1.0f / kO); };
  auto pack = [&](int o, int p) {
    const __half2 v = __floats2half2_rn(at(o, p), at(o + 1, p));
    return *reinterpret_cast<const uint32_t*>(&v);
  };
  uint4 r;
  r.x = pack(2 * t, g);       r.y = pack(2 * t + 8, g);          // n-tile 0: p = g
  r.z = pack(2 * t, 8 + g);   r.w = pack(2 * t + 8, 8 + g);      // n-tile 1: p = 8 + g
  frag[(size_t)blockIdx.x * 32 + lane] = r;
}

constexpr int kFiberGroup = 16;                                   // atoms per tile (the M of the mma)
constexpr int kFiberRowBytes = kC * kO * 2 + 16;                  // one atom's [c][o] fp16 block + 16 B: conflict-free fragment loads
constexpr int kFiberTileBytes = kFiberGroup * kFiberRowBytes;
constexpr size_t kFiberSmem = (size_t)kFiberTileBytes + (size_t)kFiberMmaWarps * 32 * 16 * sizeof(float) +
                              3 * kC * sizeof(float) + 64;      // 84 KB: two CTAs per SM

__global__ void __launch_bounds__(kFiberMmaWarps * 32, 2)
fiber_norm_mma_kernel(const __half* __restrict__ x1t, const uint4* __restrict__ fk_frag, const float* __restrict__ bias,
                      const float* __restrict__ ln_w, const float* __restrict__ ln_b, int N, __half* __restrict__ y,
                      float* __restrict__ x2_dbg) {
  // Persistent CTAs of 8 warps, two per SM (one loads while the other computes); a tile = 16 atoms (64 KB of x1t,
  // contiguous) arrives by bulk copies; warp w owns channels 16 w .. 16 w + 15 of the tile.  The B fragments (64 KB
  // per layer, the same for every tile) are read through L1.
  extern __shared__ __align__(128) uint8_t fsm[];
  const uint4* __restrict__ s_frag = fk_frag;                                    // [kC][32], L1 resident
  uint8_t* s_a = fsm;                                                            // [16 atoms][kFiberRowBytes]
  float* s_stats = reinterpret_cast<float*>(s_a + (size_t)kFiberTileBytes);      // [warps][32 lanes][16]
  float* s_bias = s_stats + kFiberMmaWarps * 32 * 16;
  float* s_g = s_bias + kC;
  float* s_b = s_g + kC;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_b + kC);                        // full
  for (int i = threadIdx.x; i < kC; i += blockDim.x) { s_bias[i] = bias[i]; s_g[i] = ln_w[i]; s_b[i] = ln_b[i]; }
  if (threadIdx.x == 0) {
    tc::mbar_init(&bars[0], 1);
    tc::fence_barrier_init();
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int groups = (N + kFiberGroup - 1) / kFiberGroup;
  auto issue = [&](int grp) {                 // thread 0: the valid atoms of tile grp
    const int atom0 = grp * kFiberGroup;
    const int n = min(kFiberGroup, N - atom0);
    tc::mbar_expect_tx(&bars[0], (uint32_t)n * (kC * kO * 2));
    for (int a = 0; a < n; ++a)
      tc::bulk_g2s(s_a + (size_t)a * kFiberRowBytes, x1t + (size_t)(atom0 + a) * kC * kO, kC * kO * 2, &bars[0]);
  };
  int it = 0;
  for (int grp = blockIdx.x; grp < groups; grp += gridDim.x, ++it) {
    if (threadIdx.x == 0) {                   // the buffer was released by the barrier that ended the previous tile
      tc::fence_proxy_async();
      issue(grp);
    }
    tc::mbar_wait(&bars[0], it & 1);
    const int atom0 = grp * kFiberGroup;
    const bool v0 = atom0 + g < N, v1 = atom0 + g + 8 < N;
    const uint8_t* a0p = s_a + (size_t)g * kFiberRowBytes + 4 * t;
    const uint8_t* a1p = a0p + 8 * (size_t)kFiberRowBytes;
    auto load_a = [&](int c, uint32_t (&a)[4]) {
      a[0] = *reinterpret_cast<const uint32_t*>(a0p + c * (kO * 2));
      a[1] = *reinterpret_cast<const uint32_t*>(a1p + c * (kO * 2));
      a[2] = *reinterpret_cast<const uint32_t*>(a0p + c * (kO * 2) + 16);
      a[3] = *reinterpret_cast<const uint32_t*>(a1p + c * (kO * 2) + 16);
    };
    // pass 1: partial statistics over this warp's 16 channels of the 8 (atom, p) pairs of the lane
    // pair index = ntile * 4 + {(g, 2t), (g, 2t+1), (g+8, 2t), (g+8, 2t+1)}
    float sum[8], sq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { sum[i] = 0.f; sq[i] = 0.f; }
#pragma unroll 4
    for (int cc = 0; cc < kC / kFiberMmaWarps; ++cc) {
      const int c = warp * (kC / kFiberMmaWarps) + cc;
      uint32_t a[4];
      load_a(c, a);
      const uint4 b = __ldg(s_frag + c * 32 + lane);
      float d0[4], d1[4];
      mma16816(d0, a[0], a[1], a[2], a[3], b.x, b.y);
      mma16816(d1, a[0], a[1], a[2], a[3], b.z, b.w);
      const float bc = s_bias[c];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float x0 = d0[i] + bc, x1v = d1[i] + bc;
        sum[i] += x0; sq[i] = fmaf(x0, x0, sq[i]);
        sum[4 + i] += x1v; sq[4 + i] = fmaf(x1v, x1v, sq[4 + i]);
      }
    }
    {
      float4* st = reinterpret_cast<float4*>(s_stats + ((size_t)warp * 32 + lane) * 16);
      st[0] = make_float4(sum[0], sum[1], sum[2], sum[3]);
      st[1] = make_float4(sum[4], sum[5], sum[6], sum[7]);
      st[2] = make_float4(sq[0], sq[1], sq[2], sq[3]);
      st[3] = make_float4(sq[4], sq[5], sq[6], sq[7]);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) { sum[i] = 0.f; sq[i] = 0.f; }
#pragma unroll
    for (int w = 0; w < kFiberMmaWarps; ++w) {      // fixed order: deterministic
      const float4* st = reinterpret_cast<const float4*>(s_stats + ((size_t)w * 32 + lane) * 16);
      const float4 s0 = st[0], s1 = st[1], q0 = st[2], q1 = st[3];
      sum[0] += s0.x; sum[1] += s0.y; sum[2] += s0.z; sum[3] += s0.w;
      sum[4] += s1.x; sum[5] += s1.y; sum[6] += s1.z; sum[7] += s1.w;
      sq[0] += q0.x; sq[1] += q0.y; sq[2] += q0.z; sq[3] += q0.w;
      sq[4] += q1.x; sq[5] += q1.y; sq[6] += q1.z; sq[7] += q1.w;
    }
    float rstd[8], shift[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float mean = sum[i] * (1.0f / kC);
      const float var = fmaxf(sq[i] * (1.0f / kC) - mean * mean, 0.f);      // biased variance, eps 1e-5 (convnext.py:25)
      rstd[i] = 1.0f / sqrtf(var + 1e-5f);
      shift[i] = -mean * rstd[i];
    }
    // pass 2: recompute, normalise, emit 16-byte chunks (8 channels) of the y tile image
    // row of pair i: (atom0 + g + 8 * ((i >> 1) & 1)) * 16 + p,  p = 8 * (i >> 2) + 2 t + (i & 1)
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int cb = warp * 2 + half;
      uint32_t pk[8][4];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        float o0[8], o1[8];
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int c = cb * 8 + j + jj;
          uint32_t a[4];
          load_a(c, a);
          const uint4 b = __ldg(s_frag + c * 32 + lane);
          float d0[4], d1[4];
          mma16816(d0, a[0], a[1], a[2], a[3], b.x, b.y);
          mma16816(d1, a[0], a[1], a[2], a[3], b.z, b.w);
          const float bc = s_bias[c], gw = s_g[c], gb = s_b[c];
          float* o = jj ? o1 : o0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float x0 = d0[i] + bc, x1v = d1[i] + bc;
            if (x2_dbg) {
              const int at0 = atom0 + g + 8 * ((i >> 1) & 1);
              if (at0 < N) {
                x2_dbg[((size_t)at0 * kO + 2 * t + (i & 1)) * kC + c] = x0;
                x2_dbg[((size_t)at0 * kO + 8 + 2 * t + (i & 1)) * kC + c] = x1v;
              }
            }
            o[i] = fmaf(fmaf(x0, rstd[i], shift[i]), gw, gb);
            o[4 + i] = fmaf(fmaf(x1v, rstd[4 + i], shift[4 + i]), gw, gb);
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __half2 v = __floats2half2_rn(o0[i], o1[i]);
          pk[i][j >> 1] = *reinterpret_cast<const uint32_t*>(&v);
        }
      }
      const int slab = cb >> 3, chunk = cb & 7;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool valid = ((i >> 1) & 1) ? v1 : v0;
        if (valid) {
          const long long row = (long long)(atom0 + g + 8 * ((i >> 1) & 1)) * kO + 8 * (i >> 2) + 2 * t + (i & 1);
          const int rr = (int)(row & 127);
          *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(y) + (size_t)(row >> 7) * 32768 + (size_t)slab * 16384 +
                                    (size_t)rr * 128 + ((chunk ^ (rr & 7)) << 4)) = make_uint4(pk[i][0], pk[i][1], pk[i][2], pk[i][3]);
        }
      }
    }
    __syncthreads();       // every warp is done with this tile's buffer and the statistics scratch
  }
}

// K4b + K5 + LayerNorm fused (fp16 path): the message sums never leave the SM.  Persistent CTAs of 8 warps, two per SM;
// per 16-atom tile a CTA alternates between two phases and the co-resident CTAs (and the other SMs) drift out of phase,
// so the HBM-bound gather of one overlaps the latency-bound tensor-core fiber conv of another:
//   phase 1  warp w gathers atoms 2w, 2w+1 of the tile: lane = 4 channels, orientations in pairs, 8 edges (16
//            independent 8/16-byte loads per lane) in flight, edges in CSR order (deterministic, no atomics); the
//            fp16 sums go to shared memory as the A operand [atom][c][o] of the fiber conv
//   phase 2  fiber_norm_mma_kernel's two passes on that tile (statistics, then recompute + normalise + emit the
//            ConvNext kernel's UMMA operand image)
// Shared-memory rows: a channel's 16 orientations are 32 contiguous bytes; 16 bytes of padding after every 4 channels
// (one lane's 128 bytes) and per atom keep both the gather's stores and the mma fragment loads conflict-free.
constexpr int kFusedWarps = 8;
constexpr int kFusedRowBytes = kC * kO * 2 + (kC / 4) * 16 + 16;              // 4624
constexpr int kFusedTileBytes = kFiberGroup * kFusedRowBytes;
constexpr size_t kFusedSmem = (size_t)kFusedTileBytes + (size_t)kFusedWarps * 32 * 16 * sizeof(float) + 3 * kC * sizeof(float);
constexpr int kPrefetchLead = 1;                 // gather iterations between a slab prefetch and its use

__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  const __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

__global__ void __launch_bounds__(kFusedWarps * 32, 2)
message_fiber_norm_fused_kernel(const __half* __restrict__ kern, const float* __restrict__ h,
                                const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ src,
                                const uint4* __restrict__ fk_frag, const float* __restrict__ bias,
                                const float* __restrict__ ln_w, const float* __restrict__ ln_b, int N,
                                __half* __restrict__ y, float* __restrict__ x2_dbg) {
  extern __shared__ __align__(128) uint8_t fsm[];
  uint8_t* s_a = fsm;                                                            // [16 atoms][kFusedRowBytes]
  float* s_stats = reinterpret_cast<float*>(s_a + (size_t)kFusedTileBytes);      // [warps][32 lanes][16]
  float* s_bias = s_stats + kFusedWarps * 32 * 16;
  float* s_g = s_bias + kC;
  float* s_b = s_g + kC;
  for (int i = threadIdx.x; i < kC; i += blockDim.x) { s_bias[i] = bias[i]; s_g[i] = ln_w[i]; s_b[i] = ln_b[i]; }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int groups = (N + kFiberGroup - 1) / kFiberGroup;
  const int e_last = max(row_ptr[N] - 1, 0);                   // for clamping the slab prefetch addresses
  for (int grp = blockIdx.x; grp < groups; grp += gridDim.x) {
    const int atom0 = grp * kFiberGroup;
    // first edge of this warp's first atom in the CTA's NEXT tile (slab prefetch across the tile boundary)
    const int next_node = (grp + (int)gridDim.x) * kFiberGroup + warp * 2;
    const int next_e0 = next_node < N ? __ldg(row_ptr + next_node) : e_last;
    // ---------------- phase 1: gather ----------------
#pragma unroll 1
    for (int rep = 0; rep < 2; ++rep) {
      const int a = warp * 2 + rep, node = atom0 + a;
      if (node >= N) break;                                    // rows past N are never stored (v0 / v1 below)
      const int e0 = row_ptr[node], e1 = row_ptr[node + 1];
      uint8_t* dst = s_a + (size_t)a * kFusedRowBytes + lane * 144;
      int sj0[8];                                              // sources of the first 8 edges: loaded once per atom
#pragma unroll
      for (int u = 0; u < 8; ++u) sj0[u] = e1 > e0 ? __ldg(src + min(e0 + u, e1 - 1)) : 0;
#pragma unroll 1
      for (int op = 0; op < kO / 2; ++op) {
        // both orientations of the pair at once: 32 independent loads per lane in flight
        const int o0 = 2 * op;
        {
          // The slab is streamed from HBM exactly once, so each of these iterations would wait for 16 DRAM misses.  Pull
          // the slab block of the iteration kPrefetchLead steps ahead into L2 now (a later orientation pair of this atom,
          // the warp's second atom -- its edges follow in CSR order --, or the warp's first atom of the CTA's next
          // tile): 8 edges x 512 B = one 128-byte line per lane, no registers held; the lead time turns the misses
          // into L2 hits (445 -> 405 us per launch at C2 with one step of lead, profiles/r2_ab_message_prefetch.txt).
          const int kk = rep * (kO / 2) + op + kPrefetchLead;       // iteration index within the tile (16 per warp)
          const int pe0 = kk >= kO ? next_e0 : ((kk >> 3) == rep ? e0 : e1);
          const int pe = min(pe0 + (lane >> 2), e_last);
          const char* pa = reinterpret_cast<const char*>(kern + ((size_t)pe * kO + 2 * (kk & 7)) * kC) + (lane & 3) * 128;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pa));
        }
        float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0;
        const int koff0 = (((lane >> 1) ^ o0) << 3) | ((lane & 1) << 2);
        const int koff1 = (((lane >> 1) ^ (o0 + 1)) << 3) | ((lane & 1) << 2);
        int e = e0;
        if (e1 - e0 >= 8) {
          // full first chunk (every atom under the neighbour cap): the 8 slab rows are 4 KB apart from one base pointer
          // (immediate offsets), the source rows one wide multiply each; no clamps, no per-edge predicates
          const __half* k0 = kern + ((size_t)e0 * kO + o0) * kC + koff0;
          const __half* k1 = kern + ((size_t)e0 * kO + o0 + 1) * kC + koff1;
          const float* hb = h + (size_t)o0 * kC + lane * 4;
          uint2 kv0[8], kv1[8];
          float4 hv0[8], hv1[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(kv0[u].x), "=r"(kv0[u].y) : "l"(k0 + (size_t)u * kO * kC));
            asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(kv1[u].x), "=r"(kv1[u].y) : "l"(k1 + (size_t)u * kO * kC));
            const float* hrow = hb + (size_t)(unsigned)sj0[u] * (kO * kC);
            hv0[u] = *reinterpret_cast<const float4*>(hrow);
            hv1[u] = *reinterpret_cast<const float4*>(hrow + kC);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&kv0[u].x));
            const float2 a1 = __half22float2(*reinterpret_cast<const __half2*>(&kv0[u].y));
            s0.x = fmaf(a0.x, hv0[u].x, s0.x);
            s0.y = fmaf(a0.y, hv0[u].y, s0.y);
            s0.z = fmaf(a1.x, hv0[u].z, s0.z);
            s0.w = fmaf(a1.y, hv0[u].w, s0.w);
            const float2 b0 = __half22float2(*reinterpret_cast<const __half2*>(&kv1[u].x));
            const float2 b1 = __half22float2(*reinterpret_cast<const __half2*>(&kv1[u].y));
            s1.x = fmaf(b0.x, hv1[u].x, s1.x);
            s1.y = fmaf(b0.y, hv1[u].y, s1.y);
            s1.z = fmaf(b1.x, hv1[u].z, s1.z);
            s1.w = fmaf(b1.y, hv1[u].w, s1.w);
          }
          e = e0 + 8;
        }
        for (; e < e1; e += 8) {
          uint2 kv0[8], kv1[8];
          float4 hv0[8], hv1[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int ee = min(e + u, e1 - 1);                  // clamped: loads stay in range, the tail is masked below
            const int sj = e == e0 ? sj0[u] : __ldg(src + ee);
            const __half* krow = kern + ((size_t)ee * kO + o0) * kC;
            // the slab is streamed once: keep it out of L1, which holds the fiber-kernel fragments and re-used h rows
            asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(kv0[u].x), "=r"(kv0[u].y) : "l"(krow + koff0));
            asm volatile("ld.global.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(kv1[u].x), "=r"(kv1[u].y) : "l"(krow + kC + koff1));
            const float* hrow = h + ((size_t)sj * kO + o0) * kC + lane * 4;
            hv0[u] = *reinterpret_cast<const float4*>(hrow);
            hv1[u] = *reinterpret_cast<const float4*>(hrow + kC);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            if (e + u < e1) {
              const float2 a0 = __half22float2(*reinterpret_cast<const __half2*>(&kv0[u].x));
              const float2 a1 = __half22float2(*reinterpret_cast<const __half2*>(&kv0[u].y));
              s0.x = fmaf(a0.x, hv0[u].x, s0.x);
              s0.y = fmaf(a0.y, hv0[u].y, s0.y);
              s0.z = fmaf(a1.x, hv0[u].z, s0.z);
              s0.w = fmaf(a1.y, hv0[u].w, s0.w);
              const float2 b0 = __half22float2(*reinterpret_cast<const __half2*>(&kv1[u].x));
              const float2 b1 = __half22float2(*reinterpret_cast<const __half2*>(&kv1[u].y));
              s1.x = fmaf(b0.x, hv1[u].x, s1.x);
              s1.y = fmaf(b0.y, hv1[u].y, s1.y);
              s1.z = fmaf(b1.x, hv1[u].z, s1.z);
              s1.w = fmaf(b1.y, hv1[u].w, s1.w);
            }
          }
        }
        // channel 4 lane + i, orientations (2 op, 2 op + 1): one half2 at [c][o]
        *reinterpret_cast<uint32_t*>(dst + 0 * 32 + op * 4) = pack_h2(s0.x, s1.x);
        *reinterpret_cast<uint32_t*>(dst + 1 * 32 + op * 4) = pack_h2(s0.y, s1.y);
        *reinterpret_cast<uint32_t*>(dst + 2 * 32 + op * 4) = pack_h2(s0.z, s1.z);
        *reinterpret_cast<uint32_t*>(dst + 3 * 32 + op * 4) = pack_h2(s0.w, s1.w);
      }
    }
    __syncthreads();
    // ---------------- phase 2: fiber conv + LayerNorm (see fiber_norm_mma_kernel) ----------------
    const bool v0 = atom0 + g < N, v1 = atom0 + g + 8 < N;
    const uint8_t* a0p = s_a + (size_t)g * kFusedRowBytes + 4 * t;
    const uint8_t* a1p = a0p + 8 * (size_t)kFusedRowBytes;
    auto load_a = [&](int c, uint32_t (&a)[4]) {
      const int off = c * (kO * 2) + (c >> 2) * 16;
      a[0] = *reinterpret_cast<const uint32_t*>(a0p + off);
      a[1] = *reinterpret_cast<const uint32_t*>(a1p + off);
      a[2] = *reinterpret_cast<const uint32_t*>(a0p + off + 16);
      a[3] = *reinterpret_cast<const uint32_t*>(a1p + off + 16);
    };
    float sum[8], sq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { sum[i] = 0.f; sq[i] = 0.f; }
#pragma unroll 4
    for (int cc = 0; cc < kC / kFusedWarps; ++cc) {
      const int c = warp * (kC / kFusedWarps) + cc;
      uint32_t a[4];
      load_a(c, a);
      const uint4 b = __ldg(fk_frag + c * 32 + lane);
      float d0[4], d1[4];
      mma16816(d0, a[0], a[1], a[2], a[3], b.x, b.y);
      mma16816(d1, a[0], a[1], a[2], a[3], b.z, b.w);
      const float bc = s_bias[c];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float x0 = d0[i] + bc, x1v = d1[i] + bc;
        sum[i] += x0; sq[i] = fmaf(x0, x0, sq[i]);
        sum[4 + i] += x1v; sq[4 + i] = fmaf(x1v, x1v, sq[4 + i]);
      }
    }
    {
      float4* st = reinterpret_cast<float4*>(s_stats + ((size_t)warp * 32 + lane) * 16);
      st[0] = make_float4(sum[0], sum[1], sum[2], sum[3]);
      st[1] = make_float4(sum[4], sum[5], sum[6], sum[7]);
      st[2] = make_float4(sq[0], sq[1], sq[2], sq[3]);
      st[3] = make_float4(sq[4], sq[5], sq[6], sq[7]);
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) { sum[i] = 0.f; sq[i] = 0.f; }
#pragma unroll
    for (int w = 0; w < kFusedWarps; ++w) {      // fixed order: deterministic
      const float4* st = reinterpret_cast<const float4*>(s_stats + ((size_t)w * 32 + lane) * 16);
      const float4 s0 = st[0], s1 = st[1], q0 = st[2], q1 = st[3];
      sum[0] += s0.x; sum[1] += s0.y; sum[2] += s0.z; sum[3] += s0.w;
      sum[4] += s1.x; sum[5] += s1.y; sum[6] += s1.z; sum[7] += s1.w;
      sq[0] += q0.x; sq[1] += q0.y; sq[2] += q0.z; sq[3] += q0.w;
      sq[4] += q1.x; sq[5] += q1.y; sq[6] += q1.z; sq[7] += q1.w;
    }
    float rstd[8], shift[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float mean = sum[i] * (1.0f / kC);
      const float var = fmaxf(sq[i] * (1.0f / kC) - mean * mean, 0.f);      // biased variance, eps 1e-5 (convnext.py:25)
      rstd[i] = 1.0f / sqrtf(var + 1e-5f);
      shift[i] = -mean * rstd[i];
    }
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      const int cb = warp * 2 + half;
      uint32_t pk[8][4];
#pragma unroll
      for (int j = 0; j < 8; j += 2) {
        float o0[8], o1[8];
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int c = cb * 8 + j + jj;
          uint32_t a[4];
          load_a(c, a);
          const uint4 b = __ldg(fk_frag + c * 32 + lane);
          float d0[4], d1[4];
          mma16816(d0, a[0], a[1], a[2], a[3], b.x, b.y);
          mma16816(d1, a[0], a[1], a[2], a[3], b.z, b.w);
          const float bc = s_bias[c], gw = s_g[c], gb = s_b[c];
          float* o = jj ? o1 : o0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float x0 = d0[i] + bc, x1v = d1[i] + bc;
            if (x2_dbg) {
              const int at0 = atom0 + g + 8 * ((i >> 1) & 1);
              if (at0 < N) {
                x2_dbg[((size_t)at0 * kO + 2 * t + (i & 1)) * kC + c] = x0;
                x2_dbg[((size_t)at0 * kO + 8 + 2 * t + (i & 1)) * kC + c] = x1v;
              }
            }
            o[i] = fmaf(fmaf(x0, rstd[i], shift[i]), gw, gb);
            o[4 + i] = fmaf(fmaf(x1v, rstd[4 + i], shift[4 + i]), gw, gb);
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) pk[i][j >> 1] = pack_h2(o0[i], o1[i]);
      }
      const int slab = cb >> 3, chunk = cb & 7;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const bool valid = ((i >> 1) & 1) ? v1 : v0;
        if (valid) {
          const long long row = (long long)(atom0 + g + 8 * ((i >> 1) & 1)) * kO + 8 * (i >> 2) + 2 * t + (i & 1);
          const int rr = (int)(row & 127);
          *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(y) + (size_t)(row >> 7) * 32768 + (size_t)slab * 16384 +
                                    (size_t)rr * 128 + ((chunk ^ (rr & 7)) << 4)) = make_uint4(pk[i][0], pk[i][1], pk[i][2], pk[i][3]);
        }
      }
    }
    __syncthreads();       // every warp is done with this tile's buffer and the statistics scratch
  }
}

constexpr int kFiberThreads = 512;
constexpr int kFiberStages = 3;
constexpr int kFiberNB = 2;     // nodes per pipeline stage

template <typename YT>
__device__ __forceinline__ void store_y_row(YT* __restrict__ y, size_t row, int cg, const float4& r) {
  if constexpr (sizeof(YT) == 4) {
    *reinterpret_cast<float4*>(y + row * kC + cg * 4) = r;
  } else {
    // fp16 y goes straight into the UMMA operand image of the ConvNext MLP kernel: 128-row tiles of
    // 32 KB, two 64-channel slabs of 128-byte rows, 16-byte chunks XOR-swizzled by (row & 7)
    // (csrc/tc_common.cuh), so that kernel fetches a tile with one bulk copy.
    const int rr = (int)(row & 127), c0 = cg * 4;
    uint8_t* tile = reinterpret_cast<uint8_t*>(y) + (row >> 7) * 32768;
    const int off = (c0 >> 6) * 16384 + rr * 128 + (((((c0 & 63) >> 3) ^ (rr & 7)) << 4) | ((c0 & 7) << 1));
    __half2 p0 = __floats2half2_rn(r.x, r.y), p1 = __floats2half2_rn(r.z, r.w);
    uint2 raw;
    raw.x = *reinterpret_cast<unsigned*>(&p0);
    raw.y = *reinterpret_cast<unsigned*>(&p1);
    *reinterpret_cast<uint2*>(tile + off) = raw;
  }
}

template <typename XT, typename YT>
__global__ void __launch_bounds__(kFiberThreads, 1)
fiber_norm_kernel(const XT* __restrict__ x1, const float* __restrict__ fk, const float* __restrict__ bias,
                  const float* __restrict__ ln_w, const float* __restrict__ ln_b, int N, YT* __restrict__ y,
                  float* __restrict__ x2_dbg) {
  // kFiberNB nodes' x1 (16 x 128 values = 8 KB fp32 / 4 KB fp16 each: one 16-byte cp.async per thread) per stage
  __shared__ __align__(16) XT xs[kFiberStages][kFiberNB][kO * kC];
  constexpr int kPer16 = 16 / sizeof(XT);                     // elements per 16-byte copy
  constexpr int kCopyThreads = kO * kC / kPer16;
  const int p = threadIdx.x >> 5, cg = threadIdx.x & 31;
  float4 fkr[kO];
#pragma unroll
  for (int o = 0; o < kO; ++o) fkr[o] = __ldg(reinterpret_cast<const float4*>(fk + ((size_t)(o * kO + p)) * kC + cg * 4));
  const float4 bv = *reinterpret_cast<const float4*>(bias + cg * 4);
  const float4 gw = *reinterpret_cast<const float4*>(ln_w + cg * 4);
  const float4 gb = *reinterpret_cast<const float4*>(ln_b + cg * 4);
  constexpr float inv_o = 1.0f / kO;
  // this CTA's node groups: g = blockIdx.x, + gridDim.x, ... (group g = nodes kFiberNB*g ..)
  const int groups = (N + kFiberNB - 1) / kFiberNB;
  auto issue = [&](int k) {
    const long long g = (long long)blockIdx.x + (long long)k * gridDim.x;
    if (g < groups) {
#pragma unroll
      for (int nb = 0; nb < kFiberNB; ++nb) {
        const long long node = g * kFiberNB + nb;
        if (node < N && threadIdx.x < kCopyThreads)
          cp_async16(&xs[k % kFiberStages][nb][threadIdx.x * kPer16], x1 + (size_t)node * kO * kC + threadIdx.x * kPer16);
      }
    }
    cp_async_commit();
  };
#pragma unroll
  for (int k = 0; k < kFiberStages - 1; ++k) issue(k);
  int k = 0;
  for (int g = blockIdx.x; g < groups; g += gridDim.x, ++k) {
    cp_async_wait<kFiberStages - 2>();
    __syncthreads();                       // stage k has landed for every thread; stage k-1 is free again
    issue(k + kFiberStages - 1);
#pragma unroll 1
    for (int nb = 0; nb < kFiberNB; ++nb) {          // one node at a time: the 16 fk registers leave room for one accumulator set
      const int node = g * kFiberNB + nb;
      if (node >= N) break;
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int o = 0; o < kO; ++o) {
        float4 xv;
        if constexpr (sizeof(XT) == 4) {
          xv = *reinterpret_cast<const float4*>(&xs[k % kFiberStages][nb][o * kC + cg * 4]);
        } else {
          const uint2 raw = *reinterpret_cast<const uint2*>(&xs[k % kFiberStages][nb][o * kC + cg * 4]);
          const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
          const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
          xv = make_float4(lo.x, lo.y, hi.x, hi.y);
        }
        t.x = fmaf(xv.x, fkr[o].x, t.x);
        t.y = fmaf(xv.y, fkr[o].y, t.y);
        t.z = fmaf(xv.z, fkr[o].z, t.z);
        t.w = fmaf(xv.w, fkr[o].w, t.w);
      }
      t.x = t.x * inv_o + bv.x;
      t.y = t.y * inv_o + bv.y;
      t.z = t.z * inv_o + bv.z;
      t.w = t.w * inv_o + bv.w;
      if (x2_dbg) *reinterpret_cast<float4*>(x2_dbg + ((size_t)node * kO + p) * kC + cg * 4) = t;
      // LayerNorm over the 128 channels held by this warp (biased variance, eps 1e-5)
      const float mean = warp_sum((t.x + t.y) + (t.z + t.w)) * (1.0f / kC);
      const float dx = t.x - mean, dy = t.y - mean, dz = t.z - mean, dw = t.w - mean;
      const float var = warp_sum((dx * dx + dy * dy) + (dz * dz + dw * dw)) * (1.0f / kC);
      const float rstd = 1.0f / sqrtf(var + 1e-5f);
      store_y_row(y, (size_t)node * kO + p, cg,
                  make_float4(dx * rstd * gw.x + gb.x, dy * rstd * gw.y + gb.y, dz * rstd * gw.z + gb.z,
                              dw * rstd * gw.w + gb.w));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K6  ConvNext channel MLP (fp32 SIMT): h += layer_scale * (W2 gelu(W1 y + b1) + b2)
// ------------------------------------------------------------------------------------------------
constexpr size_t kMlpSmemFloats = 2 * (size_t)kC * kPitch + 2 * kKC * kNT;

__global__ void __launch_bounds__(kGemmThreads, 1)
convnext_mlp_simt_kernel(const float* __restrict__ y, const float* __restrict__ w1_t, const float* __restrict__ b1,
                         const float* __restrict__ w2_t, const float* __restrict__ b2,
                         const float* __restrict__ layer_scale, long long rows, float* __restrict__ h) {
  extern __shared__ __align__(16) float smem[];
  float* Ys = smem;                 // [kC][kPitch]  y tile, transposed
  float* Hs = Ys + kC * kPitch;     // [kC][kPitch]  one 128-wide slice of the hidden layer, transposed
  float* Bs = Hs + kC * kPitch;
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const long long tiles = (rows + kTM - 1) / kTM;
  float2 acc1[8][4], acc2[8][4];
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long r0 = tile * kTM;
    for (int v = tid; v < kTM * kC / 4; v += kGemmThreads) {
      const int r = v >> 5, k4 = v & 31;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + r < rows) val = *reinterpret_cast<const float4*>(y + (size_t)(r0 + r) * kC + k4 * 4);
      Ys[(k4 * 4 + 0) * kPitch + r] = val.x;
      Ys[(k4 * 4 + 1) * kPitch + r] = val.y;
      Ys[(k4 * 4 + 2) * kPitch + r] = val.z;
      Ys[(k4 * 4 + 3) * kPitch + r] = val.w;
    }
    __syncthreads();
    zero_acc(acc2);
    for (int j = 0; j < kW / kNT; ++j) {
      zero_acc(acc1);
      gemm_pass<kC>(acc1, Ys, w1_t + j * kNT, kW, Bs, tid);
#pragma unroll
      for (int j2 = 0; j2 < 8; ++j2) {
        const int n = acc_col(tx, j2);
        const float bb = b1[j * kNT + n];
        *reinterpret_cast<float4*>(Hs + n * kPitch + ty * 4) =
            make_float4(gelu_erf(acc_get(acc1, 0, j2) + bb), gelu_erf(acc_get(acc1, 1, j2) + bb),
                        gelu_erf(acc_get(acc1, 2, j2) + bb), gelu_erf(acc_get(acc1, 3, j2) + bb));
        *reinterpret_cast<float4*>(Hs + n * kPitch + 64 + ty * 4) =
            make_float4(gelu_erf(acc_get(acc1, 4, j2) + bb), gelu_erf(acc_get(acc1, 5, j2) + bb),
                        gelu_erf(acc_get(acc1, 6, j2) + bb), gelu_erf(acc_get(acc1, 7, j2) + bb));
      }
      gemm_pass<kNT>(acc2, Hs, w2_t + (size_t)j * kNT * kC, kC, Bs, tid);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const long long row = r0 + acc_row(ty, i);
      if (row < rows) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int c0 = half * 64 + tx * 4;
          float* hp = h + (size_t)row * kC + c0;
          float4 hv = *reinterpret_cast<float4*>(hp);
          const float4 bb = *reinterpret_cast<const float4*>(b2 + c0);
          const float4 ls = *reinterpret_cast<const float4*>(layer_scale + c0);
          const float2 p0 = acc2[i][half * 2], p1 = acc2[i][half * 2 + 1];
          hv.x = fmaf(ls.x, p0.x + bb.x, hv.x);
          hv.y = fmaf(ls.y, p0.y + bb.y, hv.y);
          hv.z = fmaf(ls.z, p1.x + bb.z, hv.z);
          hv.w = fmaf(ls.w, p1.y + bb.w, hv.w);
          *reinterpret_cast<float4*>(hp) = hv;
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------
// K7  read-outs.  By linearity the orientation pooling is applied before the Linear:
//   mean_o (Wr h[b,o] + br) = Wr (mean_o h[b,o]) + br.
// acc[N][Z+6] = [logits (Z) | score vector (3) | length channels (3)], summed over layers.
// ------------------------------------------------------------------------------------------------
constexpr int kReadoutNodes = 8;

__global__ void __launch_bounds__(kC)
readout_accumulate_kernel(const float* __restrict__ h, const float* __restrict__ wr_t, const float* __restrict__ br,
                          const float* __restrict__ ori, int N, int Z, int first_layer, float* __restrict__ acc) {
  __shared__ __align__(16) float hbar[kReadoutNodes][kC];   // mean over orientations
  __shared__ float s_o[kReadoutNodes][kO];                  // vector-channel read-out per orientation
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int R = Z + 4;   // read-out rows: Z scalars, 1 vector channel, 3 global scalars (ponita.py:111)
  const int b0 = blockIdx.x * kReadoutNodes;
  // phase A: one warp per atom (two atoms per warp), lane = 4 channels.  The 16 per-orientation dot products with
  // the vector-channel row are reduced across the warp with a transpose-reduce (16 values over 32 lanes:
  // 8 + 4 + 2 + 1 + 1 = 16 shuffles instead of 16 x 5).
  float4 wv;
  wv.x = wr_t[(size_t)(lane * 4 + 0) * R + Z];
  wv.y = wr_t[(size_t)(lane * 4 + 1) * R + Z];
  wv.z = wr_t[(size_t)(lane * 4 + 2) * R + Z];
  wv.w = wr_t[(size_t)(lane * 4 + 3) * R + Z];
  const float bz = br[Z];
#pragma unroll
  for (int rep = 0; rep < kReadoutNodes / 4; ++rep) {
    const int a = warp + 4 * rep, b = b0 + a;
    float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b < N) {
      const float* hp = h + (size_t)b * kO * kC + lane * 4;
      float4 hv[kO];                                    // all 16 rows in flight before the first use
#pragma unroll
      for (int o = 0; o < kO; ++o) hv[o] = __ldcs(reinterpret_cast<const float4*>(hp + o * kC));
      float d[kO];
#pragma unroll
      for (int o = 0; o < kO; ++o) {
        sum.x += hv[o].x; sum.y += hv[o].y; sum.z += hv[o].z; sum.w += hv[o].w;
        d[o] = (hv[o].x * wv.x + hv[o].y * wv.y) + (hv[o].z * wv.z + hv[o].w * wv.w);
      }
      // transpose-reduce: after the step with lane distance `dist`, a lane keeps half of its values
      // (those whose index bit matches its lane bit) summed with the partner's copy
#pragma unroll
      for (int i = 0; i < 8; ++i) {                     // distance 16: keep d[i] (lane bit 4 = 0) or d[i + 8]
        const bool up = lane & 16;
        const float send = up ? d[i] : d[i + 8];
        const float keep = up ? d[i + 8] : d[i];
        d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {                     // distance 8
        const bool up = lane & 8;
        const float send = up ? d[i] : d[i + 4];
        const float keep = up ? d[i + 4] : d[i];
        d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i) {                     // distance 4
        const bool up = lane & 4;
        const float send = up ? d[i] : d[i + 2];
        const float keep = up ? d[i + 2] : d[i];
        d[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
      }
      {                                                 // distance 2
        const bool up = lane & 2;
        const float send = up ? d[0] : d[1];
        const float keep = up ? d[1] : d[0];
        d[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
      }
      d[0] += __shfl_xor_sync(0xffffffffu, d[0], 1);    // distance 1: both lanes of a pair hold the total
      // this lane now holds orientation o = 8 b4 + 4 b3 + 2 b2 + b1 of its lane bits
      if ((lane & 1) == 0) s_o[a][((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)] = d[0] + bz;
    }
    constexpr float inv = 1.0f / kO;
    *reinterpret_cast<float4*>(&hbar[a][lane * 4]) = make_float4(sum.x * inv, sum.y * inv, sum.z * inv, sum.w * inv);
  }
  __syncthreads();
  // phase B: thread z owns read-out row z for the CTA's atoms (each weight load is reused for all of them)
  if (tid < R && tid != Z) {
    const int z = tid;
    float r[kReadoutNodes];
    const float bb = br[z];
#pragma unroll
    for (int a = 0; a < kReadoutNodes; ++a) r[a] = bb;
    for (int k = 0; k < kC; ++k) {
      const float w = wr_t[(size_t)k * R + z];
#pragma unroll
      for (int a = 0; a < kReadoutNodes; ++a) r[a] = fmaf(w, hbar[a][k], r[a]);
    }
    const int slot = z < Z ? z : (Z + 3 + (z - Z - 1));
#pragma unroll
    for (int a = 0; a < kReadoutNodes; ++a)
      if (b0 + a < N) {
        float* p = acc + (size_t)(b0 + a) * (Z + 6) + slot;
        *p = first_layer ? r[a] : *p + r[a];
      }
  } else if (tid >= R && tid < R + 3 * kReadoutNodes && tid - R < 3 * kReadoutNodes) {
    const int a = (tid - R) / 3, d = (tid - R) % 3;
    if (b0 + a < N) {
      float sacc = 0.f;
#pragma unroll
      for (int o = 0; o < kO; ++o) sacc = fmaf(s_o[a][o], ori[3 * o + d], sacc);   // to_from_sphere.py:10-11
      sacc *= (1.0f / kO);
      float* p = acc + (size_t)(b0 + a) * (Z + 6) + Z + d;
      *p = first_layer ? sacc : *p + sacc;
    }
  }
}

// Pooled read-out of all layers in one pass (fp16 tensor path).  pool[k], k = 0..L, holds the orientation-pooled features
// after the embedding (k = 0, node_embed_kernel) and the pooled residual UPDATE of interaction layer k (k = 1..L, pool
// warps of convnext_mlp_tc_kernel), as [group of 16 atoms][4 parts][C][16 atoms] with parts
// [mean_o . | (1/O) sum_o ori[o][d] ., d = 0..2].  The read-out Linear commutes with the pooling
// (to_from_sphere.py:10-14) and the feature after layer l is the sum of entries 0..l, so
//   mean_l read_out_l(h_l) = sum_k V_k pool[k] + bias,   V_k = (1/L) sum_{l >= max(k,1)} Wr_l
// with V_k[C][96] and bias[96] combined once on the host (weights.py) in the column layout of acc[N][Z+6]:
// columns 0..Z-1 logits, Z..Z+2 the score vector (weight row Z applied to parts 1..3), Z+3..Z+5 length channels.
// One persistent CTA per SM; per entry k the 48 KB matrix sits in shared memory; a warp owns a group of 16 atoms:
// lane = output columns (lane, lane + 32, lane + 64), 16 atoms x 3 columns accumulated as packed FFMA2 over atom pairs;
// the group's pooled block streams through a per-warp cp.async double buffer in chunks of 32 channels; acc is updated
// in place in a fixed order (deterministic).
constexpr int kPoolAtoms = 16;
constexpr int kPoolCols = 96;
constexpr int kPoolWarps = 8;
// One pool entry = [groups][C][16 atoms] of the orientation mean, then [groups * 16 atoms][8] partial contractions of
// the vector-pooled parts with the score row: element 2 d + half (d = 0..2; the producer's two channel halves).
// One persistent CTA per SM; per entry k the 48 KB matrix V_k sits in shared memory; a warp owns a group of 16 atoms:
// lane = output columns (lane, lane + 32, lane + 64), 16 atoms x 3 columns accumulated as packed FFMA2 over atom pairs
// (fp32 throughout: the read-outs feed the D3PM argmax and the coordinate update directly); the group's 8 KB block
// arrives through a per-warp cp.async double buffer (the next group's block is in flight while this one is
// multiplied); lanes 0..15 add the producers' score partials of one atom each; acc is updated in place, entry by entry,
// in a fixed order (deterministic).  (A mma.sync TF32 version with the 3xTF32 split measured 0.26 ms against this
// kernel's FFMA2: the legacy tensor path delivers ~70 TFLOP/s of TF32 on this part, a third of that after the split.)
constexpr int kRpBlockFloats = kC * kPoolAtoms;                                 // 2048 floats = 8 KB
constexpr int kRpSmem = (kC * kPoolCols + kPoolWarps * 2 * kRpBlockFloats) * (int)sizeof(float);

__global__ void __launch_bounds__(kPoolWarps * 32, 1)
readout_pooled_kernel(const float* __restrict__ pool, size_t entry_stride, const float* __restrict__ v,
                      const float* __restrict__ bias, int N, int Z, int entries, float* __restrict__ acc) {
  extern __shared__ __align__(16) float rp_sm[];
  float* const vs = rp_sm;                                                       // [kC][kPoolCols]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* const pb = rp_sm + kC * kPoolCols + warp * 2 * kRpBlockFloats;          // this warp's [2][C][16 atoms]
  const int groups = (N + kPoolAtoms - 1) / kPoolAtoms;
  // columns Z..Z+2 (the score vector) come from the producers' partials, not from this product
  const int col2 = lane + 64;
  const bool skip2 = col2 >= Z && col2 < Z + 3;
  auto load_block = [&](const float* gsrc, int buf) {                            // 8 KB, 16 bytes per lane and copy
    float* dst = pb + buf * kRpBlockFloats;
#pragma unroll
    for (int i = 0; i < kRpBlockFloats / 128; ++i) cp_async16(dst + (i * 32 + lane) * 4, gsrc + (i * 32 + lane) * 4);
    cp_async_commit();
  };
  for (int k = 0; k < entries; ++k) {
    __syncthreads();                                                             // the previous matrix is no longer read
    for (int i = tid; i < kC * kPoolCols / 4; i += kPoolWarps * 32)
      reinterpret_cast<float4*>(vs)[i] = __ldg(reinterpret_cast<const float4*>(v + (size_t)k * kC * kPoolCols) + i);
    __syncthreads();
    const float* entry = pool + (size_t)k * entry_stride;
    const float* partials = entry + (size_t)groups * kRpBlockFloats;
    const int g0 = blockIdx.x * kPoolWarps + warp, gstep = gridDim.x * kPoolWarps;
    if (g0 < groups) load_block(entry + (size_t)g0 * kRpBlockFloats, 0);
    auto load_acc = [&](int base, float2 (&x)[3][kPoolAtoms / 2]) {              // running sums of a group (bias at k = 0)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const bool skip = j == 2 && skip2;
        const float bb = k == 0 ? bias[lane + 32 * j] : 0.f;
#pragma unroll
        for (int a = 0; a < kPoolAtoms / 2; ++a) {
          const int a0 = base + 2 * a;
          x[j][a].x = k == 0 ? bb : ((a0 < N && !skip) ? acc[(size_t)a0 * kPoolCols + lane + 32 * j] : 0.f);
          x[j][a].y = k == 0 ? bb : ((a0 + 1 < N && !skip) ? acc[(size_t)(a0 + 1) * kPoolCols + lane + 32 * j] : 0.f);
        }
      }
    };
    float2 rn[3][kPoolAtoms / 2];
    int it = 0;
    for (int grp = g0; grp < groups; grp += gstep, ++it) {
      const int b0 = grp * kPoolAtoms;
      if (grp + gstep < groups) {
        load_block(entry + (size_t)(grp + gstep) * kRpBlockFloats, (it + 1) & 1);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncwarp();
      float2 r[3][kPoolAtoms / 2];
      if (it == 0) load_acc(b0, r);
      else {
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
          for (int a = 0; a < kPoolAtoms / 2; ++a) r[j][a] = rn[j][a];
      }
      // the next group's running sums are fetched now, under this group's products
      if (grp + gstep < groups) load_acc(b0 + gstep * kPoolAtoms, rn);
      // score vector (columns Z..Z+2): lanes 0..15 own one atom each and add the producers' partial contractions
      float sc[3] = {0.f, 0.f, 0.f};
      const bool sv = lane < kPoolAtoms && b0 + lane < N;
      if (sv) {
        const float4 s0 = __ldg(reinterpret_cast<const float4*>(partials + (size_t)(b0 + lane) * 8));
        const float4 s1 = __ldg(reinterpret_cast<const float4*>(partials + (size_t)(b0 + lane) * 8) + 1);
        const float* prev = acc + (size_t)(b0 + lane) * kPoolCols + Z;
        sc[0] = (k == 0 ? bias[Z] : prev[0]) + (s0.x + s0.y);
        sc[1] = (k == 0 ? bias[Z + 1] : prev[1]) + (s0.z + s0.w);
        sc[2] = (k == 0 ? bias[Z + 2] : prev[2]) + (s1.x + s1.y);
      }
      const float* p0 = pb + (it & 1) * kRpBlockFloats;
      const float* w = vs + lane;
#pragma unroll 2
      for (int c = 0; c < kC; ++c) {
        const float w0 = w[c * kPoolCols], w1 = w[c * kPoolCols + 32], w2 = w[c * kPoolCols + 64];
        const float2 w0d = make_float2(w0, w0), w1d = make_float2(w1, w1), w2d = make_float2(w2, w2);
#pragma unroll
        for (int q4 = 0; q4 < kPoolAtoms / 4; ++q4) {
          const float4 pa = *reinterpret_cast<const float4*>(p0 + c * kPoolAtoms + 4 * q4);
          const float2 pa0 = make_float2(pa.x, pa.y), pa1 = make_float2(pa.z, pa.w);
          r[0][2 * q4] = __ffma2_rn(w0d, pa0, r[0][2 * q4]);
          r[0][2 * q4 + 1] = __ffma2_rn(w0d, pa1, r[0][2 * q4 + 1]);
          r[1][2 * q4] = __ffma2_rn(w1d, pa0, r[1][2 * q4]);
          r[1][2 * q4 + 1] = __ffma2_rn(w1d, pa1, r[1][2 * q4 + 1]);
          r[2][2 * q4] = __ffma2_rn(w2d, pa0, r[2][2 * q4]);
          r[2][2 * q4 + 1] = __ffma2_rn(w2d, pa1, r[2][2 * q4 + 1]);
        }
      }
      __syncwarp();                                                              // the buffer is refilled by the next iteration
#pragma unroll
      for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int a = 0; a < kPoolAtoms / 2; ++a) {
          const int a0 = b0 + 2 * a;
          const bool skip = j == 2 && skip2;
          if (a0 < N && !skip) acc[(size_t)a0 * kPoolCols + lane + 32 * j] = r[j][a].x;
          if (a0 + 1 < N && !skip) acc[(size_t)(a0 + 1) * kPoolCols + lane + 32 * j] = r[j][a].y;
        }
      if (sv) {
        float* o = acc + (size_t)(b0 + lane) * kPoolCols + Z;
        o[0] = sc[0]; o[1] = sc[1]; o[2] = sc[2];
      }
    }
  }
}

__global__ void readout_finalize_kernel(const float* __restrict__ acc, const int32_t* __restrict__ atom_offset, int N,
                                        int G, int Z, float inv_layers, float* __restrict__ logits,
                                        float* __restrict__ score, float* __restrict__ len0) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long n_node = (long long)N * (Z + 3);
  if (idx < n_node) {
    const int b = (int)(idx / (Z + 3)), k = (int)(idx % (Z + 3));
    const float v = acc[(size_t)b * (Z + 6) + k] * inv_layers;
    if (k < Z) logits[(size_t)b * Z + k] = v;
    else score[(size_t)b * 3 + (k - Z)] = v;
  } else if (idx < n_node + 3LL * G) {
    const int g = (int)((idx - n_node) / 3), d = (int)((idx - n_node) % 3);
    float s = 0.f;   // global_add_pool (ponita.py:152): fixed atom order
    for (int b = atom_offset[g]; b < atom_offset[g + 1]; ++b) s += acc[(size_t)b * (Z + 6) + Z + 3 + d] * inv_layers;
    len0[3 * g + d] = s;
  }
}

int num_sms() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
static int node_embed_launch(const float* x, const float* vec, const float* w_embed_t, const float* ori,
                             const int64_t* types, int32_t Z, int32_t N, int32_t F, int32_t V, float* h, float* pool,
                             const float* pool_wz, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!x || !vec || !w_embed_t || !ori || !h) return ARREAU_ERR_NULL;
  if (N < 0 || F <= 0 || V < 0 || V > kMaxVec || (types && (Z <= 0 || Z > F))) return ARREAU_ERR_BAD_SHAPE;
  size_t smem = sizeof(float) * ((size_t)kEmbedNodes * (F + V * kO) + (size_t)kEmbedNodes * V * 4 + 4);
  if (pool && smem < sizeof(float) * kEmbedNodes * kC) smem = sizeof(float) * kEmbedNodes * kC;
  if (smem > 48 * 1024) return ARREAU_ERR_UNSUPPORTED;
  if (V == 4)
    node_embed_kernel<4><<<(N + kEmbedNodes - 1) / kEmbedNodes, kEmbedNodes * 32, smem, (cudaStream_t)stream>>>(
        x, vec, w_embed_t, ori, types, Z, N, F, V, h, pool, pool_wz, Z);
  else
    node_embed_kernel<0><<<(N + kEmbedNodes - 1) / kEmbedNodes, kEmbedNodes * 32, smem, (cudaStream_t)stream>>>(
        x, vec, w_embed_t, ori, types, Z, N, F, V, h, pool, pool_wz, Z);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_node_embed(const float* x, const float* vec, const float* w_embed_t, const float* ori,
                                 int32_t N, int32_t F, int32_t V, float* h, void* stream) {
  return node_embed_launch(x, vec, w_embed_t, ori, nullptr, 0, N, F, V, h, nullptr, nullptr, stream);
}

extern "C" int arreau_node_embed_typed(const float* x, const int64_t* types, int32_t Z, const float* vec,
                                       const float* w_embed_t, const float* ori, int32_t N, int32_t F, int32_t V,
                                       float* h, void* stream) {
  if (!types) return ARREAU_ERR_NULL;
  return node_embed_launch(x, vec, w_embed_t, ori, types, Z, N, F, V, h, nullptr, nullptr, stream);
}

extern "C" int arreau_node_embed_pooled(const float* x, const int64_t* types, int32_t Z, const float* vec,
                                        const float* w_embed_t, const float* ori, int32_t N, int32_t F, int32_t V,
                                        float* h, float* pool, const float* readout_v0, void* stream) {
  if (N > 0 && (!pool || !readout_v0)) return ARREAU_ERR_NULL;
  if (Z + 6 != 96) return ARREAU_ERR_UNSUPPORTED;
  return node_embed_launch(x, vec, w_embed_t, ori, types, Z, N, F, V, h, pool, readout_v0, stream);
}

extern "C" int arreau_fiber_kernel_precompute(const float* ori, const float* w1, const float* b1, const float* w2,
                                              const float* b2, const float* wf, float* fiber_kernel, void* stream) {
  if (!ori || !w1 || !b1 || !w2 || !b2 || !wf || !fiber_kernel) return ARREAU_ERR_NULL;
  fiber_kernel_kernel<<<kO * kO, kD, 0, (cudaStream_t)stream>>>(ori, w1, b1, w2, b2, wf, fiber_kernel);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_edge_kernels_f32(const double* dir, const double* dist, const double* lattice,
                                       const int32_t* crystal_of_atom, const int32_t* src,
                                       const int32_t* num_edges_ptr, int64_t edge_capacity, const float* ori,
                                       const float* w1m_t, const float* w2_t, const float* b2, const float* wk_t,
                                       double radius, float* kernels, void* stream) {
  if (edge_capacity == 0) return ARREAU_OK;
  if (!dir || !dist || !lattice || !crystal_of_atom || !src || !num_edges_ptr || !ori || !w1m_t || !w2_t || !b2 ||
      !wk_t || !kernels)
    return ARREAU_ERR_NULL;
  if (edge_capacity < 0) return ARREAU_ERR_BAD_SHAPE;
  static bool attr_set = false;
  const size_t smem = kEdgeSmemFloats * sizeof(float);
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(edge_kernels_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const long long tiles = (edge_capacity + kEdgesPerTile - 1) / kEdgesPerTile;
  const int grid = (int)(tiles < (long long)num_sms() ? tiles : (long long)num_sms());
  edge_kernels_simt_kernel<<<grid, kGemmThreads, smem, (cudaStream_t)stream>>>(
      dir, dist, lattice, crystal_of_atom, src, num_edges_ptr, (long long)edge_capacity, ori, w1m_t, w2_t, b2, wk_t,
      radius, kernels);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_fiber_frag_pack(const float* fiber_kernel, int32_t num_layers, void* fiber_frag, void* stream) {
  if (!fiber_kernel || !fiber_frag) return ARREAU_ERR_NULL;
  if (num_layers <= 0) return ARREAU_ERR_BAD_SHAPE;
  fiber_frag_kernel<<<num_layers * kC, 32, 0, (cudaStream_t)stream>>>(fiber_kernel, (uint4*)fiber_frag);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_message_gather(const void* kernels, int32_t kernels_f16, const float* h, const int32_t* row_ptr,
                                     const int32_t* src, int32_t N, int32_t x1_f16_transposed, float* x1, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!h || !row_ptr || !x1 || !kernels) return ARREAU_ERR_NULL;
  if (N < 0 || (x1_f16_transposed && !kernels_f16)) return ARREAU_ERR_BAD_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  const long long rows = (long long)N * kO;
  if (x1_f16_transposed) {
    message_gather_t_kernel<<<N, kGatherTThreads, 0, s>>>((const __half*)kernels, h, row_ptr, src, N, (__half*)x1);
  } else {
    const unsigned ggrid = (unsigned)((rows + kGatherWarps - 1) / kGatherWarps);
    if (kernels_f16)
      message_gather_kernel<__half, float><<<ggrid, kGatherWarps * 32, 0, s>>>((const __half*)kernels, h, row_ptr, src, rows, x1);
    else
      message_gather_kernel<float, float><<<ggrid, kGatherWarps * 32, 0, s>>>((const float*)kernels, h, row_ptr, src, rows, x1);
  }
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_fiber_norm(const float* x1, int32_t x1_f16_transposed, const float* fiber_kernel,
                                 const void* fiber_frag, const float* conv_bias, const float* ln_w, const float* ln_b,
                                 int32_t N, void* y, int32_t y_f16, float* x2_debug, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!x1 || !fiber_kernel || !conv_bias || !ln_w || !ln_b || !y) return ARREAU_ERR_NULL;
  if (N < 0 || (x1_f16_transposed && !y_f16)) return ARREAU_ERR_BAD_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  if (x1_f16_transposed) {
    if (!fiber_frag) return ARREAU_ERR_NULL;
    static bool attr_set = false;
    if (!attr_set) {
      cudaError_t e = cudaFuncSetAttribute(fiber_norm_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFiberSmem);
      if (e != cudaSuccess) return (int)e;
      attr_set = true;
    }
    const int groups = (N + kFiberGroup - 1) / kFiberGroup;
    const int grid = groups < 2 * num_sms() ? groups : 2 * num_sms();
    fiber_norm_mma_kernel<<<grid, kFiberMmaWarps * 32, kFiberSmem, s>>>((const __half*)x1, (const uint4*)fiber_frag, conv_bias,
                                                                        ln_w, ln_b, N, (__half*)y, x2_debug);
  } else {
    const int fgroups = (N + kFiberNB - 1) / kFiberNB;
    const int fgrid = fgroups < num_sms() ? fgroups : num_sms();
    if (y_f16)
      fiber_norm_kernel<float, __half><<<fgrid, kFiberThreads, 0, s>>>(x1, fiber_kernel, conv_bias, ln_w, ln_b, N, (__half*)y, x2_debug);
    else
      fiber_norm_kernel<float, float><<<fgrid, kFiberThreads, 0, s>>>(x1, fiber_kernel, conv_bias, ln_w, ln_b, N, (float*)y, x2_debug);
  }
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_message_fiber_norm_fused(const void* kernels_f16, const float* h, const int32_t* row_ptr,
                                               const int32_t* src, const void* fiber_frag, const float* conv_bias,
                                               const float* ln_w, const float* ln_b, int32_t N, void* y_f16,
                                               float* x2_debug, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!kernels_f16 || !h || !row_ptr || !src || !fiber_frag || !conv_bias || !ln_w || !ln_b || !y_f16) return ARREAU_ERR_NULL;
  if (N < 0) return ARREAU_ERR_BAD_SHAPE;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(message_fiber_norm_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFusedSmem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const int groups = (N + kFiberGroup - 1) / kFiberGroup;
  const int grid = groups < 2 * num_sms() ? groups : 2 * num_sms();
  message_fiber_norm_fused_kernel<<<grid, kFusedWarps * 32, kFusedSmem, (cudaStream_t)stream>>>(
      (const __half*)kernels_f16, h, row_ptr, src, (const uint4*)fiber_frag, conv_bias, ln_w, ln_b, N, (__half*)y_f16, x2_debug);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_message_fiber_norm(const void* kernels, int32_t kernels_f16, const float* h,
                                         const int32_t* row_ptr, const int32_t* src, const float* fiber_kernel,
                                         const void* fiber_frag, const float* conv_bias, const float* ln_w,
                                         const float* ln_b, int32_t N, void* y, int32_t y_f16, float* x1,
                                         float* x2_debug, void* stream) {
  // fp16 tensor path (fp16 kernels in, fp16 y out): ONE fused launch, the message sums stay in shared memory
  const int32_t t = (kernels_f16 && y_f16) ? 1 : 0;
  if (t) return arreau_message_fiber_norm_fused(kernels, h, row_ptr, src, fiber_frag, conv_bias, ln_w, ln_b, N, y, x2_debug, stream);
  const int rc = arreau_message_gather(kernels, kernels_f16, h, row_ptr, src, N, t, x1, stream);
  if (rc != ARREAU_OK) return rc;
  return arreau_fiber_norm(x1, t, fiber_kernel, fiber_frag, conv_bias, ln_w, ln_b, N, y, y_f16, x2_debug, stream);
}

extern "C" int arreau_convnext_mlp_f32(const float* y, const float* w1_t, const float* b1, const float* w2_t,
                                       const float* b2, const float* layer_scale, int64_t num_rows, float* h,
                                       void* stream) {
  if (num_rows == 0) return ARREAU_OK;
  if (!y || !w1_t || !b1 || !w2_t || !b2 || !layer_scale || !h) return ARREAU_ERR_NULL;
  if (num_rows < 0) return ARREAU_ERR_BAD_SHAPE;
  static bool attr_set = false;
  const size_t smem = kMlpSmemFloats * sizeof(float);
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(convnext_mlp_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const long long tiles = (num_rows + kTM - 1) / kTM;
  const int grid = (int)(tiles < (long long)num_sms() ? tiles : (long long)num_sms());
  convnext_mlp_simt_kernel<<<grid, kGemmThreads, smem, (cudaStream_t)stream>>>(y, w1_t, b1, w2_t, b2, layer_scale,
                                                                                (long long)num_rows, h);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_readout_accumulate(const float* h, const float* wr_t, const float* br, const float* ori,
                                         int32_t N, int32_t Z, int32_t first_layer, float* acc, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!h || !wr_t || !br || !ori || !acc) return ARREAU_ERR_NULL;
  if (N < 0 || Z <= 0) return ARREAU_ERR_BAD_SHAPE;
  if (Z + 4 + 3 * kReadoutNodes > kC) return ARREAU_ERR_UNSUPPORTED;
  readout_accumulate_kernel<<<(N + kReadoutNodes - 1) / kReadoutNodes, kC, 0, (cudaStream_t)stream>>>(h, wr_t, br, ori, N,
                                                                                                    Z, first_layer, acc);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_readout_pooled(const float* pool, const float* readout_v, const float* readout_bias, int32_t N,
                                     int32_t Z, int32_t entries, float* acc, void* stream) {
  if (N == 0) return ARREAU_OK;
  if (!pool || !readout_v || !readout_bias || !acc) return ARREAU_ERR_NULL;
  if (N < 0 || entries <= 0) return ARREAU_ERR_BAD_SHAPE;
  if (Z + 6 != kPoolCols) return ARREAU_ERR_UNSUPPORTED;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(readout_pooled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kRpSmem);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const int groups = (N + kPoolAtoms - 1) / kPoolAtoms;
  const int ctas = (groups + kPoolWarps - 1) / kPoolWarps;
  const int grid = ctas < num_sms() ? ctas : num_sms();
  readout_pooled_kernel<<<grid, kPoolWarps * 32, kRpSmem, (cudaStream_t)stream>>>(
      pool, (size_t)groups * 4 * kC * kPoolAtoms, readout_v, readout_bias, N, Z, entries, acc);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_readout_finalize(const float* acc, const int32_t* atom_offset, int32_t N, int32_t G, int32_t Z,
                                       int32_t num_layers, float* logits, float* score, float* len0, void* stream) {
  if (N == 0 && G == 0) return ARREAU_OK;
  if (!acc || !atom_offset || !logits || !score || !len0) return ARREAU_ERR_NULL;
  if (N < 0 || G < 0 || Z <= 0 || num_layers <= 0) return ARREAU_ERR_BAD_SHAPE;
  const long long total = (long long)N * (Z + 3) + 3LL * G;
  readout_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      acc, atom_offset, N, G, Z, 1.0f / (float)num_layers, logits, score, len0);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}
