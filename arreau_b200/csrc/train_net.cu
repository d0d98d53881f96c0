// Training step of the Ponita fiber-bundle network (SURVEY 8a rows a19-a23) on sm_100a: the hand-derived backward pass
// and, in TF32 mode, the training forward that keeps what the backward needs.
//
// The reference obtains parameter gradients with torch autograd through
//   ponita/models/ponita.py:88-155, ponita/nn/conv.py:105-133, ponita/nn/convnext.py:20-33,
//   ponita/nn/embedding.py:4-14, ponita/utils/windowing.py:21-29, ponita/utils/to_from_sphere.py:4-14
// (inputs carry no gradient: positions, lattice and the graph are data).  Here the same derivatives are
// written out by hand as a fixed sequence of kernels on one stream:
//
//   * every dense contraction (kept or recomputed activations, input gradients, weight gradients) goes through ONE
//     generic GEMM that reads either operand in either storage order, so that the parameters and their gradients stay
//     in the reference's own state_dict layouts ([out, in] row-major) with no transposed copies.  Three kernels behind it:
//       sgemm_kernel      fp32 SIMT (128x128x16 tiles, packed FFMA2): ARREAU_PRECISION_FP32, the parity path;
//       sgemm_tma_kernel  ARREAU_PRECISION_TF32: persistent, warp-specialised tcgen05 kind::tf32 kernel fed by TMA tensor
//                         maps, double-buffered TMEM accumulators, fused epilogues (bias, GELU, GELU', residual, column
//                         sums) -- see the comment above it;
//       sgemm_tc_kernel   the same product one tile per CTA with register-staged operands: the TF32 path for operands a
//                         tensor map cannot describe (K < 32, ragged contiguous extents); gemm() picks it from the
//                         operands alone;
//   * weight gradients reduce over the rows (edges x orientations, or atoms x orientations): split-K with
//     per-split partial tiles and a fixed-order second stage -- no atomics, bit-reproducible run to run;
//   * the message pass is transposed with a sender-side gather in edge order (deterministic) instead of
//     scatter atomics; the same pass writes the sender's rows of the kernel gradient.
//
// The forward pass of a training step is either the ordinary fp32 forward (arreau_ponita_forward) run with its per-layer
// buffers kept (h, x1, x2 of every layer and the per-layer spatial kernels; the backward then recomputes the rest), or
// arreau_ponita_forward_train below (TF32 mode): the same mathematics with its dense contractions on the generic GEMM
// and every activation the backward reads kept in the backward's workspace.
#include <cuda.h>          // CUtensorMap and its enums only: cuTensorMapEncodeTiled is reached through the runtime

#include "common.cuh"
#include "tc_common.cuh"

namespace {

// ================================================================================================
// generic fp32 GEMM   C[M,N] (=|+=) alpha * A x B (+ bias[n])
//   AK: A stored [M][K] (K contiguous, row pitch lda)   else [K][M] (M contiguous)
//   BK: B stored [N][K] (K contiguous, row pitch ldb)   else [K][N] (N contiguous)
// grid = (ceil(N/128), ceil(M/128), splits); with splits > 1 the raw tile sums go to
// partial[split][M][N] and sgemm_reduce_kernel finishes (alpha, bias, accumulate).
// Requirements: K-contiguous operands need K % 4 == 0 and pitch % 4 == 0; the other storage order needs
// the contiguous extent % 4 == 0; pointers 16-byte aligned.
// ================================================================================================
constexpr int kBM = 128, kBN = 128, kBK = 16, kSP = 132, kGT = 256;

// One GEMM launch.  Every matrix is addressed through a ROW PITCH (ld*) over its strided index and a BLOCK STRIDE (*_cblk)
// over 128-element blocks of its contiguous index: element i of the contiguous index lives at (i >> 7) * cblk + (i & 127).
// cblk = 128 is the ordinary dense matrix; another value strings together equally shaped slabs that are 128 wide each --
// the per-layer [rows][128] kernel / kernel-gradient slabs of the five layers act as ONE [rows][640] (or [640][rows]) operand
// or output, so the five per-layer products of conv.py:110 (and their two transposes in the backward) are one launch each
// and the shared operand is streamed from HBM once instead of five times.
// Epilogue (unsplit launches only), in this order:  v = alpha * acc + bias[n];  v *= gelu'(gz[m][n]) * rowscale[m >> 4]  (gz);
// v += C (accumulate);  C = v;  C2 = gelu(v) * rowscale[m >> 4]  (C2: the activation next to its pre-activation, so that no
// separate element-wise pass re-reads the matrix), or, with res_in:  C2 = res_in + res_scale[n] * v  (the residual update
// of the ConvNext block next to the kept MLP output).
struct GemmArgs {
  const float* A; long long lda, a_cblk;
  const float* B; long long ldb, b_cblk;
  float* C; long long ldc, c_cblk;
  int M, N; long long K, k_per_split;
  float alpha; const float* bias; int accumulate;
  float* partial;
  float* C2;
  const float* gz; long long gz_ld;
  const float* rowscale;
  const float* res_in; const float* res_scale;   // C2 = res_in[m][n] + res_scale[n] * v (pitch ldc) instead of the GELU
  int splits;                 // K splits (the persistent kernel's grid is not the tile grid)
  float* colsum_part;         // persistent kernel: per-CTA column sums of C, [grid / ntn * 4][N] (see GemmOpt::colsum_out), or null
  long long* prof;            // debug: per-CTA phase clocks of the persistent kernel ([grid][16]), or null
};

__device__ __forceinline__ long long blk_off(long long i, long long cblk) { return (i >> 7) * cblk + (i & 127); }

__device__ __forceinline__ float gelu_grad(float x) {
  // d/dx [0.5 x (1 + erf(x / sqrt 2))] = 0.5 (1 + erf(x / sqrt 2)) + x exp(-x^2 / 2) / sqrt(2 pi)
  return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * expf(-0.5f * x * x) * 0.39894228040143267794f;
}

// GELU and its derivative for the TF32 kernels' epilogues, where the exact erff / expf pair (~60 instructions per value)
// made the fused epilogues the bound of the HBM-bound products: Phi(x) = 1/2 erfc(-x / sqrt 2) from the Abramowitz-Stegun
// 7.1.26 rational form (absolute error 1.5e-7, no cancellation on the negative side) and ONE ex2.approx shared by Phi and
// the density: exp(-x^2 / 2) is both erfc's factor and sqrt(2 pi) phi(x).
__device__ __forceinline__ void gelu_parts_fast(float x, float& cdf, float& e) {
  const float a = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, a, 1.0f));
  e = __expf(-a * a);
  const float h = 0.5f * e * t * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 1.061405429f, -1.453152027f), 1.421413741f), -0.284496736f), 0.254829592f);
  cdf = x < 0.f ? h : 1.0f - h;
}
template <bool FAST>
__device__ __forceinline__ float gelu_fwd_t(float x) {
  if (!FAST) return gelu_erf(x);
  float cdf, e;
  gelu_parts_fast(x, cdf, e);
  return x * cdf;
}
template <bool FAST>
__device__ __forceinline__ float gelu_grad_t(float x) {
  if (!FAST) return gelu_grad(x);
  float cdf, e;
  gelu_parts_fast(x, cdf, e);
  return fmaf(x * 0.39894228040143267794f, e, cdf);
}

// the four accumulators (m, n .. n + 3) of a tile on their way out (n % 4 == 0, n < N)
template <bool FAST = false>
__device__ __forceinline__ float4 gemm_store4(const GemmArgs& g, bool split, int z, int m, int n, float4 v,
                                              const float4* gz_loaded = nullptr) {
  if (split) {
    *reinterpret_cast<float4*>(g.partial + ((size_t)z * g.M + m) * g.N + n) = v;
    return v;
  }
  float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
  if (g.bias) bb = *reinterpret_cast<const float4*>(g.bias + n);
  v.x = fmaf(v.x, g.alpha, bb.x); v.y = fmaf(v.y, g.alpha, bb.y); v.z = fmaf(v.z, g.alpha, bb.z); v.w = fmaf(v.w, g.alpha, bb.w);
  const float rs = g.rowscale ? g.rowscale[m >> 4] : 1.0f;
  if (g.gz) {
    const float4 z = gz_loaded ? *gz_loaded : *reinterpret_cast<const float4*>(g.gz + (long long)m * g.gz_ld + n);
    v.x *= gelu_grad_t<FAST>(z.x) * rs; v.y *= gelu_grad_t<FAST>(z.y) * rs;
    v.z *= gelu_grad_t<FAST>(z.z) * rs; v.w *= gelu_grad_t<FAST>(z.w) * rs;
  }
  const long long off = (long long)m * g.ldc + blk_off(n, g.c_cblk);
  if (g.accumulate) {
    const float4 c = *reinterpret_cast<const float4*>(g.C + off);
    v.x += c.x; v.y += c.y; v.z += c.z; v.w += c.w;
  }
  *reinterpret_cast<float4*>(g.C + off) = v;
  if (g.res_in) {
    const float4 r = *reinterpret_cast<const float4*>(g.res_in + off), sc = *reinterpret_cast<const float4*>(g.res_scale + n);
    *reinterpret_cast<float4*>(g.C2 + off) = make_float4(fmaf(sc.x, v.x, r.x), fmaf(sc.y, v.y, r.y), fmaf(sc.z, v.z, r.z), fmaf(sc.w, v.w, r.w));
  } else if (g.C2)
    *reinterpret_cast<float4*>(g.C2 + off) = make_float4(gelu_fwd_t<FAST>(v.x) * rs, gelu_fwd_t<FAST>(v.y) * rs,
                                                         gelu_fwd_t<FAST>(v.z) * rs, gelu_fwd_t<FAST>(v.w) * rs);
  return v;      // what went to C
}

template <bool KCONTIG>
__device__ __forceinline__ void tile_fetch(const float* __restrict__ X, long long ld, long long cblk, int x0, int xext,
                                           long long k0, long long kend, int tid, float4 (&r)[2]) {
  // KCONTIG: X[x][k]: float4 v -> x = v >> 2, k = (v & 3) * 4 ; else X[k][x]: v -> k = v >> 5, x = (v & 31) * 4
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int v = tid + u * kGT;
    r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KCONTIG) {
      const int x = x0 + (v >> 2);
      const long long k = k0 + (v & 3) * 4;
      if (x < xext && k < kend) r[u] = __ldg(reinterpret_cast<const float4*>(X + (long long)x * ld + blk_off(k, cblk)));
    } else {
      const long long k = k0 + (v >> 5);
      const int x = x0 + (v & 31) * 4;
      if (k < kend && x < xext) r[u] = __ldg(reinterpret_cast<const float4*>(X + k * ld + blk_off(x, cblk)));
    }
  }
}

__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}

template <bool KCONTIG>
__device__ __forceinline__ void tile_stage(float* __restrict__ S, int tid, const float4 (&r)[2]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int v = tid + u * kGT;
    const float4 q = r[u];
    if (KCONTIG) {
      const int x = v >> 2, k = (v & 3) * 4;
      S[(k + 0) * kSP + x] = q.x;
      S[(k + 1) * kSP + x] = q.y;
      S[(k + 2) * kSP + x] = q.z;
      S[(k + 3) * kSP + x] = q.w;
    } else {
      const int k = v >> 5, x = (v & 31) * 4;
      *reinterpret_cast<float4*>(S + k * kSP + x) = q;
    }
  }
}

template <bool AK, bool BK>
__global__ void __launch_bounds__(kGT)
sgemm_kernel(const __grid_constant__ GemmArgs g) {
  __shared__ __align__(16) float As[2][kBK * kSP];
  __shared__ __align__(16) float Bs[2][kBK * kSP];
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * kBN;
  const int M = g.M, N = g.N;
  const long long kbeg = (long long)blockIdx.z * g.k_per_split;
  const long long kend = (kbeg + g.k_per_split < g.K) ? kbeg + g.k_per_split : g.K;
  float2 acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = make_float2(0.f, 0.f);
  float4 ra[2], rb[2];
  if (kbeg < kend) {
    tile_fetch<AK>(g.A, g.lda, g.a_cblk, m0, M, kbeg, kend, tid, ra);
    tile_fetch<BK>(g.B, g.ldb, g.b_cblk, n0, N, kbeg, kend, tid, rb);
    tile_stage<AK>(As[0], tid, ra);
    tile_stage<BK>(Bs[0], tid, rb);
  }
  __syncthreads();
  int buf = 0;
  for (long long k0 = kbeg; k0 < kend; k0 += kBK) {
    const bool more = k0 + kBK < kend;
    if (more) {
      tile_fetch<AK>(g.A, g.lda, g.a_cblk, m0, M, k0 + kBK, kend, tid, ra);
      tile_fetch<BK>(g.B, g.ldb, g.b_cblk, n0, N, k0 + kBK, kend, tid, rb);
    }
    const float* a = As[buf];
    const float* b = Bs[buf];
#pragma unroll
    for (int k = 0; k < kBK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(a + k * kSP + ty * 4);
      const float4 a1 = *reinterpret_cast<const float4*>(a + k * kSP + 64 + ty * 4);
      const float4 b0 = *reinterpret_cast<const float4*>(b + k * kSP + tx * 4);
      const float4 b1 = *reinterpret_cast<const float4*>(b + k * kSP + 64 + tx * 4);
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
    if (more) {
      tile_stage<AK>(As[buf ^ 1], tid, ra);
      tile_stage<BK>(Bs[buf ^ 1], tid, rb);
    }
    __syncthreads();
    buf ^= 1;
  }
  const bool split = gridDim.z > 1;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int m = m0 + ((i < 4) ? (ty * 4 + i) : (64 + ty * 4 + i - 4));
    if (m >= M) continue;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int n = n0 + half * 64 + tx * 4;
      if (n >= N) continue;
      gemm_store4(g, split, (int)blockIdx.z, m, n,
                  make_float4(acc[i][half * 2].x, acc[i][half * 2].y, acc[i][half * 2 + 1].x, acc[i][half * 2 + 1].y));
    }
  }
}

// ================================================================================================
// tcgen05 variant of the same GEMM (ARREAU_PRECISION_TF32 on sm_100a): kind::tf32 UMMA, fp32 accumulation in TMEM.
//   * one 128 x 128 output tile per CTA (grid as above), K in slabs of 32 (one 128-byte swizzle row of fp32);
//   * operands go global -> registers -> shared memory (rounded to TF32 with cvt.rna on the way, as the mma.sync
//     version did) straight into the layout the UMMA descriptor reads, WITHOUT transposing:
//       K-contiguous storage  X[x][k]  -> canonical K-major  SWIZZLE_128B tile: row x = 128 B, 8-row groups 1 KB apart
//       MN-contiguous storage X[k][x]  -> canonical MN-major tile in the one layout tcgen05 accepts for 32-bit MN-major
//                                         operands, SWIZZLE_128B_BASE32B: atom = 32 x-elements (128 B) x 4 k, the 32-byte
//                                         chunk c of k-row j at chunk position c ^ j; 4 atoms along x (LBO = 512 B),
//                                         8 along k (SBO = 2 KB); a_major / b_major = 1
//     so the weight-gradient GEMMs (both operands row-major over the reduced rows) need no transposed copies either;
//   * 3-stage ring of 32 KB stages, all 8 warps load (next slab's global loads in flight under the current slab's
//     stores and the barrier), warp 0 issues the slab's four 128x128x8 MMAs warp-uniformly with one elected lane and
//     commits the stage's "empty" barrier; two CTAs per SM overlap one's loads with the other's MMAs;
//   * epilogue: tcgen05.ld, then alpha / bias / accumulate or the split-K partial tile as in the kernels above.
// Requirements as above (K % 4, pitches % 4, 16-byte aligned pointers); M, N arbitrary (zero-filled tiles), N % 4 == 0.
// ================================================================================================
namespace tcg {
constexpr int kStages = 3;
constexpr int kSlab = 32;                        // K per stage: one 128-byte row of fp32
constexpr int kOperandBytes = 128 * 128;         // 128 (M or N) x 32 K x 4 B
constexpr int kStageBytes = 2 * kOperandBytes;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 + 128;
__host__ __device__ constexpr uint32_t idesc_tf32(bool a_mn, bool b_mn) {
  // c_format F32 (bit 4), a_format / b_format TF32 = 2 (bits 7.., 10..), a_major / b_major (bits 15, 16: 1 = MN-major),
  // N >> 3 at bit 17, M >> 4 at bit 24
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32_e(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                            uint32_t idesc, uint32_t elected, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
      "setp.ne.u32 e, %6, 0;\n\t"
      "setp.ne.u32 p, %7, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %5, p;\n\t}"
      ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(elected), "r"(accumulate)
      : "memory");
}
}  // namespace tcg

template <bool KCONTIG>
__device__ __forceinline__ void tc_fetch(const float* __restrict__ X, long long ld, long long cblk, int x0, int xext,
                                         long long k0, long long kend, int tid, float4 (&r)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int v = tid + u * kGT;
    r[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KCONTIG) {                       // X[x][k]: v -> row x = v >> 3, 16-byte chunk (4 k) = v & 7
      const int x = x0 + (v >> 3);
      const long long k = k0 + (v & 7) * 4;
      if (x < xext && k < kend) r[u] = __ldg(reinterpret_cast<const float4*>(X + (long long)x * ld + blk_off(k, cblk)));
    } else {                             // X[k][x]: v -> k = v >> 5, 4 x-elements = v & 31
      const long long k = k0 + (v >> 5);
      const int x = x0 + (v & 31) * 4;
      if (k < kend && x < xext) r[u] = __ldg(reinterpret_cast<const float4*>(X + k * ld + blk_off(x, cblk)));
    }
  }
}

// L2 prefetch of one operand's slab (128 lines of 128 B) by 128 threads (t = 0..127): the register-staged loaders keep
// only ONE slab in flight per CTA, so without it every slab of a streamed operand costs a full DRAM round trip
// (measured 5.6 K cycles per slab on the step's skinny shapes); prefetched two slabs ahead the loads hit L2.
template <bool KCONTIG>
__device__ __forceinline__ void tc_prefetch(const float* __restrict__ X, long long ld, long long cblk, int x0, int xext,
                                            long long k0, long long kend, int t) {
  const float* p = nullptr;
  if (KCONTIG) {                       // X[x][k]: one line = the 32 k of row x0 + t
    if (x0 + t < xext && k0 < kend) p = X + (long long)(x0 + t) * ld + blk_off(k0, cblk);
  } else {                             // X[k][x]: 4 lines per k row
    const long long k = k0 + (t >> 2);
    const int x = x0 + (t & 3) * 32;
    if (k < kend && x < xext) p = X + k * ld + blk_off(x, cblk);
  }
  if (p) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

template <bool KCONTIG>
__device__ __forceinline__ void tc_stage(uint8_t* __restrict__ tile, int tid, const float4 (&r)[4]) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int v = tid + u * kGT;
    const float4 q = make_float4(to_tf32(r[u].x), to_tf32(r[u].y), to_tf32(r[u].z), to_tf32(r[u].w));
    uint32_t off;
    if (KCONTIG) {
      const int row = v >> 3, chunk = v & 7;
      off = (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4));
    } else {
      const int kk = v >> 5, x4 = v & 31, j = kk & 3;
      off = (uint32_t)((kk >> 2) * 2048 + (x4 >> 3) * 512 + j * 128 + (((((x4 & 7) >> 1) ^ j) << 5) | ((x4 & 1) << 4)));
    }
    *reinterpret_cast<float4*>(tile + off) = q;
  }
}

template <bool AK, bool BK>
__global__ void __launch_bounds__(kGT, 2)
sgemm_tc_kernel(const __grid_constant__ GemmArgs g) {
  using namespace tc;
  const float* __restrict__ A = g.A;
  const float* __restrict__ B = g.B;
  const long long lda = g.lda, ldb = g.ldb, K = g.K, k_per_split = g.k_per_split;
  const int M = g.M, N = g.N;
  extern __shared__ __align__(1024) uint8_t gsm_raw[];
  const uint32_t base = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  uint8_t* const sm = gsm_raw + (base - smem_u32(gsm_raw));
  uint64_t* const bar_empty = reinterpret_cast<uint64_t*>(sm + tcg::kStages * tcg::kStageBytes);   // [kStages]
  uint64_t* const bar_done = bar_empty + tcg::kStages;
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bar_done + 1);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int m0 = blockIdx.y * kBM, n0 = blockIdx.x * kBN;
  const long long kbeg = (long long)blockIdx.z * k_per_split;
  const long long kend = (kbeg + k_per_split < K) ? kbeg + k_per_split : K;
  const int nslabs = kbeg < kend ? (int)((kend - kbeg + tcg::kSlab - 1) / tcg::kSlab) : 0;
  if (tid == 0) {
    for (int i = 0; i < tcg::kStages; ++i) mbar_init(&bar_empty[i], 1);
    mbar_init(bar_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  const uint32_t el = warp == 0 ? elect_one() : 0u;
  constexpr uint32_t kIdesc = tcg::idesc_tf32(!AK, !BK);
  // descriptor words: K-major: LBO unused (1), SBO = 1 KB (8-row groups), SWIZZLE_128B; MN-major: LBO = stride between the
  // 32-element atoms along M/N, SBO = stride between the 4-k atoms (tc_stage's layout), SWIZZLE_128B_BASE32B; version 1
  constexpr int mn_lbo = 512, mn_sbo = 2048;
  const uint32_t hi_k = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
  const uint32_t hi_mn = (uint32_t)(mn_sbo >> 4) | (1u << 14) | (1u << 29);      // layout type 1 = SWIZZLE_128B_BASE32B
  const uint32_t a_hi = AK ? hi_k : hi_mn, b_hi = BK ? hi_k : hi_mn;
  const uint32_t a_lbo = AK ? (1u << 16) : ((uint32_t)(mn_lbo >> 4) << 16), b_lbo = BK ? (1u << 16) : ((uint32_t)(mn_lbo >> 4) << 16);
  constexpr uint32_t a_kstep = AK ? 2u : (4096u >> 4), b_kstep = BK ? 2u : (4096u >> 4);   // +8 K per MMA

  float4 ra[4], rb[4];
  constexpr int kPrefetchAhead = 3;            // slabs of L2 prefetch lead
  if (nslabs > 0) {
    tc_fetch<AK>(A, lda, g.a_cblk, m0, M, kbeg, kend, tid, ra);
    tc_fetch<BK>(B, ldb, g.b_cblk, n0, N, kbeg, kend, tid, rb);
#pragma unroll
    for (int a = 1; a < kPrefetchAhead; ++a) {
      const long long kp = kbeg + (long long)a * tcg::kSlab;
      if (tid < 128) tc_prefetch<AK>(A, lda, g.a_cblk, m0, M, kp, kend, tid);
      else tc_prefetch<BK>(B, ldb, g.b_cblk, n0, N, kp, kend, tid - 128);
    }
  }
  for (int s = 0; s < nslabs; ++s) {
    {
      const long long kp = kbeg + (long long)(s + kPrefetchAhead) * tcg::kSlab;
      if (tid < 128) tc_prefetch<AK>(A, lda, g.a_cblk, m0, M, kp, kend, tid);
      else tc_prefetch<BK>(B, ldb, g.b_cblk, n0, N, kp, kend, tid - 128);
    }
    const int stage = s % tcg::kStages;
    if (s >= tcg::kStages) mbar_wait(&bar_empty[stage], (uint32_t)((s / tcg::kStages - 1) & 1));   // its MMAs have read it
    uint8_t* const ta = sm + stage * tcg::kStageBytes;
    uint8_t* const tb = ta + tcg::kOperandBytes;
    tc_stage<AK>(ta, tid, ra);
    tc_stage<BK>(tb, tid, rb);
    fence_proxy_async();                        // generic-proxy stores -> visible to the UMMA operand reads
    if (s + 1 < nslabs) {                       // next slab's loads fly under the barrier and the MMA issue
      const long long k0 = kbeg + (long long)(s + 1) * tcg::kSlab;
      tc_fetch<AK>(A, lda, g.a_cblk, m0, M, k0, kend, tid, ra);
      tc_fetch<BK>(B, ldb, g.b_cblk, n0, N, k0, kend, tid, rb);
    }
    __syncthreads();
    if (warp == 0) {
      tc_fence_after();
      const uint32_t a_lo = ((smem_u32(ta) & 0x3FFFFu) >> 4) | a_lbo, b_lo = ((smem_u32(tb) & 0x3FFFFu) >> 4) | b_lbo;
#pragma unroll
      for (int ki = 0; ki < 4; ++ki)
        tcg::umma_tf32_e(tmem, a_lo + ki * a_kstep, a_hi, b_lo + ki * b_kstep, b_hi, kIdesc, el, (s > 0 || ki > 0) ? 1u : 0u);
      umma_commit_e(smem_u32(&bar_empty[stage]), el);
      if (s + 1 == nslabs) umma_commit_e(smem_u32(bar_done), el);
    }
  }
  // ---- epilogue: TMEM -> registers -> shared memory (row pitch 132 floats: conflict-free 16-byte stores of 32 rows) ->
  // coalesced 512-byte row segments to global (a thread owns ONE row of the accumulator, so writing it out directly
  // would touch 32 different rows per store instruction) ----
  const int q = warp & 3, half = warp >> 2;
  const bool split = gridDim.z > 1;
  constexpr int kPitch = 132;
  float* const stage = reinterpret_cast<float*>(sm);          // 128 x 132 floats = 66 KB of the (now idle) ring
  if (nslabs > 0) {
    mbar_wait(bar_done, 0);                                    // every MMA has completed: accumulators final, ring idle
    tc_fence_after();
  }
  {
    float* srow = stage + (q * 32 + lane) * kPitch + half * 64;
#pragma unroll
    for (int part = 0; part < 4; ++part) {
      uint32_t r[16];
      if (nslabs > 0) {
        tmem_ld16(tmem + ((uint32_t)(q * 32) << 16) + half * 64 + part * 16, r);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = 0u;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(srow + part * 16 + j * 4) = make_uint4(r[4 * j], r[4 * j + 1], r[4 * j + 2], r[4 * j + 3]);
    }
  }
  tc_fence_before();
  __syncthreads();
  {
    const int n = n0 + lane * 4;
    for (int r = warp; r < kBM; r += kGT / 32) {
      const int m = m0 + r;
      if (m >= M || n >= N) continue;
      gemm_store4(g, split, (int)blockIdx.z, m, n, *reinterpret_cast<const float4*>(stage + r * kPitch + lane * 4));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 128);
  }
}

// ================================================================================================
// The same product as a PERSISTENT, WARP-SPECIALISED kernel fed by the TMA engine (the default of ARREAU_PRECISION_TF32).
// The step's products are skinny (285 k rows x 128 .. 640 columns, K = 128 .. 640) and HBM-bound; with one tile per CTA and
// every warp loading, then multiplying, then storing, each CTA is a serial chain of memory round trips (2 .. 3 TB/s), and a
// persistent kernel whose warps copy with cp.async is bound by the SM's load/store pipe instead (1.4 K cycles of issue per
// 32 KB slab + 0.9 K for rounding it in place: profiles/r2_gemm_cpasync_phases.txt).  Here one CTA per SM walks over the work
// items (m tile, n tile, K split; n fastest, so that the SMs working side by side share the rows of A in L2):
//   warp 0      producer: one thread issues two cp.async.bulk.tensor loads per slab (tensor maps built per launch on the
//               host, data type TFLOAT32: the TMA engine rounds fp32 -> TF32 on the way, so no thread touches the operands),
//               hardware swizzle straight into the UMMA tile images, up to kStages slabs in flight across tile boundaries:
//                 K-contiguous storage  X[x][k]: box 32 k x 128 rows, SWIZZLE_128B           -> K-major tile (as above)
//                 MN-contiguous storage X[k][x]: box 32 x * 32 k * 4 atoms, SWIZZLE_128B_ATOM_32B -> MN-major tile with the
//                 atoms 4 KB apart (LBO) and the 4-k groups 512 B apart (SBO);
//               block-strided operands (GemmArgs) get one more tensor dimension;
//   warp 1      MMA issue: four 128x128x8 kind::tf32 MMAs per slab, tcgen05.commit -> empty[stage]; the accumulator is
//               double-buffered in tensor memory (2 x 128 columns), commit -> tmem_full[buffer] after a tile's last slab;
//   warps 2-17  epilogue: warp w owns TMEM lanes 32 (w % 4) and 32 columns: tcgen05.ld, release of the buffer (tmem_empty),
//               then through a private shared-memory staging tile, so that the global stores (and the loads of the fused
//               epilogue, GemmArgs) are whole 128-byte row segments; GELU / GELU' in the fast form above.
// So the loads of tile i + 1, the MMAs of tile i and the stores of tile i - 1 overlap.
// ================================================================================================
namespace wsg {
constexpr int kStages = 4;
constexpr int kMmaWarp = 1;
constexpr int kEpiWarps = 16;
constexpr int kThreads = (2 + kEpiWarps) * 32;
constexpr int kStagePitch = 36;                  // floats: 32 columns + 4 (conflict-free 16-byte rows)
constexpr int kStagingBytes = kEpiWarps * 32 * kStagePitch * 4;
constexpr int kSmemBytes = kStages * tcg::kStageBytes + kStagingBytes + 256 + 1024;
constexpr int kMnLbo = 4096, kMnSbo = 512;       // MN-major tile image written by the TMA box (see above)
}  // namespace wsg

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
               ::"r"(dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
// one 128 x 32 operand slab: x0 = first row / column of the tile, k = first K index (a multiple of 32)
template <bool KCONTIG>
__device__ __forceinline__ void tma_slab(uint32_t dst, const CUtensorMap* m, uint32_t bar, bool blocked, int x0, long long k) {
  if (KCONTIG) {
    if (!blocked) tma_load_2d(dst, m, bar, (int)k, x0);
    else tma_load_3d(dst, m, bar, (int)(k & 127), x0, (int)(k >> 7));
  } else {
    if (!blocked) tma_load_3d(dst, m, bar, 0, (int)k, x0 >> 5);
    else tma_load_4d(dst, m, bar, 0, (int)k, 0, x0 >> 7);
  }
}

// a work item of the persistent kernel (shared by the three roles)
struct WsItem {
  int m0, n0, z, nslabs;
  long long kbeg, kend;
};
__device__ __forceinline__ WsItem ws_item(const GemmArgs& g, int item, int ntn, int ntm) {
  WsItem w;
  const int nt = item % ntn, r = item / ntn;
  w.n0 = nt * kBN;
  w.m0 = (r % ntm) * kBM;
  w.z = r / ntm;
  w.kbeg = (long long)w.z * g.k_per_split;
  w.kend = (w.kbeg + g.k_per_split < g.K) ? w.kbeg + g.k_per_split : g.K;
  w.nslabs = w.kbeg < w.kend ? (int)((w.kend - w.kbeg + tcg::kSlab - 1) / tcg::kSlab) : 0;
  return w;
}

long long* g_ws_prof = nullptr;   // debug: see GemmArgs::prof

template <bool AK, bool BK>
__global__ void __launch_bounds__(wsg::kThreads, 1)
sgemm_tma_kernel(const __grid_constant__ GemmArgs g, const __grid_constant__ CUtensorMap map_a,
                 const __grid_constant__ CUtensorMap map_b) {
  using namespace tc;
  extern __shared__ __align__(1024) uint8_t gsm_raw[];
  const uint32_t base = (smem_u32(gsm_raw) + 1023u) & ~1023u;
  uint8_t* const sm = gsm_raw + (base - smem_u32(gsm_raw));
  float* const staging = reinterpret_cast<float*>(sm + wsg::kStages * tcg::kStageBytes);
  uint64_t* const bar_full = reinterpret_cast<uint64_t*>(sm + wsg::kStages * tcg::kStageBytes + wsg::kStagingBytes);
  uint64_t* const bar_empty = bar_full + wsg::kStages;
  uint64_t* const bar_tfull = bar_empty + wsg::kStages;     // [2]
  uint64_t* const bar_tempty = bar_tfull + 2;               // [2]
  uint32_t* const tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const int ntn = (g.N + kBN - 1) / kBN, ntm = (g.M + kBM - 1) / kBM;
  const int items = ntn * ntm * g.splits;
  if (tid == 0) {
    for (int i = 0; i < wsg::kStages; ++i) {
      mbar_init(&bar_full[i], 1);
      mbar_init(&bar_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar_tfull[i], 1);
      mbar_init(&bar_tempty[i], wsg::kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == wsg::kMmaWarp) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  long long pf[3] = {0, 0, 0}, t0 = clock64(), t1;
#define WS_PROF(i) { t1 = clock64(); pf[i] += t1 - t0; t0 = t1; }

  if (warp == 0) {
    // ---------------- producer ----------------
    if (lane == 0) {
      const bool a_blocked = g.a_cblk != 128, b_blocked = g.b_cblk != 128;
      uint32_t slab = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const WsItem w = ws_item(g, item, ntn, ntm);
        for (int s = 0; s < w.nslabs; ++s, ++slab) {
          const uint32_t st = slab % wsg::kStages;
          WS_PROF(1)
          if (slab >= (uint32_t)wsg::kStages) mbar_wait(&bar_empty[st], ((slab / wsg::kStages) - 1) & 1);
          WS_PROF(0)
          const uint32_t ta = base + st * tcg::kStageBytes, bar = smem_u32(&bar_full[st]);
          const long long k = w.kbeg + (long long)s * tcg::kSlab;
          mbar_expect_tx(&bar_full[st], tcg::kStageBytes);
          tma_slab<AK>(ta, &map_a, bar, a_blocked, w.m0, k);
          tma_slab<BK>(ta + tcg::kOperandBytes, &map_b, bar, b_blocked, w.n0, k);
        }
      }
      WS_PROF(1)
      if (g.prof) {
        long long* o = g.prof + (size_t)blockIdx.x * 16;
        o[0] = pf[0]; o[1] = pf[1]; o[2] = slab;
      }
    }
  } else if (warp == wsg::kMmaWarp) {
    // ---------------- MMA issue ----------------
    const uint32_t el = elect_one();
    constexpr uint32_t kIdesc = tcg::idesc_tf32(!AK, !BK);
    const uint32_t hi_k = (uint32_t)(1024 >> 4) | (1u << 14) | (2u << 29);
    const uint32_t hi_mn = (uint32_t)(wsg::kMnSbo >> 4) | (1u << 14) | (1u << 29);   // layout type 1 = SWIZZLE_128B_BASE32B
    const uint32_t a_hi = AK ? hi_k : hi_mn, b_hi = BK ? hi_k : hi_mn;
    const uint32_t a_lbo = AK ? (1u << 16) : ((uint32_t)(wsg::kMnLbo >> 4) << 16), b_lbo = BK ? (1u << 16) : ((uint32_t)(wsg::kMnLbo >> 4) << 16);
    constexpr uint32_t a_kstep = AK ? 2u : (uint32_t)(2 * wsg::kMnSbo >> 4), b_kstep = BK ? 2u : (uint32_t)(2 * wsg::kMnSbo >> 4);   // +8 K per MMA
    uint32_t slab = 0, tile = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const WsItem w = ws_item(g, item, ntn, ntm);
      if (w.nslabs == 0) continue;
      const uint32_t buf = tile & 1;
      WS_PROF(2)
      if (tile >= 2) mbar_wait(&bar_tempty[buf], ((tile >> 1) - 1) & 1);       // the epilogue has read this buffer
      WS_PROF(0)
      tc_fence_after();
      for (int s = 0; s < w.nslabs; ++s, ++slab) {
        const uint32_t st = slab % wsg::kStages;
        WS_PROF(2)
        mbar_wait(&bar_full[st], (slab / wsg::kStages) & 1);
        WS_PROF(1)
        tc_fence_after();
        const uint32_t ta = base + st * tcg::kStageBytes, tb = ta + tcg::kOperandBytes;
        const uint32_t a_lo = ((ta & 0x3FFFFu) >> 4) | a_lbo, b_lo = ((tb & 0x3FFFFu) >> 4) | b_lbo;
#pragma unroll
        for (int ki = 0; ki < 4; ++ki)
          tcg::umma_tf32_e(tmem + buf * 128, a_lo + ki * a_kstep, a_hi, b_lo + ki * b_kstep, b_hi, kIdesc, el,
                           (s > 0 || ki > 0) ? 1u : 0u);
        umma_commit_e(smem_u32(&bar_empty[st]), el);
      }
      umma_commit_e(smem_u32(&bar_tfull[buf]), el);
      ++tile;
    }
    if (g.prof && lane == 0) {
      long long* o = g.prof + (size_t)blockIdx.x * 16;
      o[3] = pf[0]; o[4] = pf[1]; o[5] = pf[2];
    }
  } else {
    // ---------------- epilogue ----------------
    const int ew = warp - wsg::kMmaWarp - 1;           // 0..15
    const int q = warp & 3, cq = ew >> 2;              // TMEM lane quarter of this warp (warp % 4), column quarter
    float* const st = staging + ew * 32 * wsg::kStagePitch;
    const bool split = g.splits > 1;
    uint32_t tile = 0;
    // fused column sums of C (bias gradients): this warp's rows of every tile of the CTA, four columns per lane (the host
    // launches this mode only when every item of a CTA has the same n tile: gridDim.x % ntn == 0)
    float4 cs = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const WsItem w = ws_item(g, item, ntn, ntm);
      const uint32_t buf = tile & 1;
      const int n = w.n0 + cq * 32 + (lane & 7) * 4;
      // the pre-activations of a fused GELU' do not depend on the product: fetched before the wait for the accumulator
      float4 gzv[8];
      if (g.gz && !split) {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int m = w.m0 + q * 32 + it * 4 + (lane >> 3);
          gzv[it] = (m < g.M && n < g.N) ? __ldg(reinterpret_cast<const float4*>(g.gz + (long long)m * g.gz_ld + n))
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
      WS_PROF(1)
      if (w.nslabs > 0) {
        mbar_wait(&bar_tfull[buf], (tile >> 1) & 1);
        tc_fence_after();
      }
      WS_PROF(0)
      {
        uint32_t r[2][16];
        if (w.nslabs > 0) {
          const uint32_t ta = tmem + ((uint32_t)(q * 32) << 16) + buf * 128 + cq * 32;
          tmem_ld16_nowait(ta, r[0]);
          tmem_ld16_nowait(ta + 16, r[1]);
          tmem_wait_ld();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bar_tempty[buf]);     // the MMAs of the tile after next may overwrite it
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) r[0][i] = r[1][i] = 0u;
        }
        float* srow = st + lane * wsg::kStagePitch;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint32_t* rr = r[j >> 2] + (j & 3) * 4;
          *reinterpret_cast<uint4*>(srow + j * 4) = make_uint4(rr[0], rr[1], rr[2], rr[3]);
        }
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int row = it * 4 + (lane >> 3);
          const int m = w.m0 + q * 32 + row;
          if (m < g.M && n < g.N) {
            const float4 v = gemm_store4<true>(g, split, w.z, m, n,
                                               *reinterpret_cast<const float4*>(st + row * wsg::kStagePitch + (lane & 7) * 4), &gzv[it]);
            cs.x += v.x; cs.y += v.y; cs.z += v.z; cs.w += v.w;
          }
        }
        __syncwarp();
      }
      if (w.nslabs > 0) ++tile;
    }
    if (g.colsum_part) {
      // the four row groups of a lane's columns (lanes l, l + 8, l + 16, l + 24), in a fixed order
#pragma unroll
      for (int off = 8; off < 32; off <<= 1) {
        cs.x += __shfl_xor_sync(0xffffffffu, cs.x, off);
        cs.y += __shfl_xor_sync(0xffffffffu, cs.y, off);
        cs.z += __shfl_xor_sync(0xffffffffu, cs.z, off);
        cs.w += __shfl_xor_sync(0xffffffffu, cs.w, off);
      }
      const int n = (int)(blockIdx.x % ntn) * kBN + cq * 32 + lane * 4;
      if (lane < 8 && n < g.N)
        *reinterpret_cast<float4*>(g.colsum_part + ((size_t)(blockIdx.x / ntn) * 4 + q) * g.N + n) = cs;
    }
    WS_PROF(1)
    if (g.prof && ew == 0 && lane == 0) {
      long long* o = g.prof + (size_t)blockIdx.x * 16;
      o[6] = pf[0]; o[7] = pf[1];
    }
  }
#undef WS_PROF
  tc_fence_before();
  __syncthreads();
  if (warp == wsg::kMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// ---- tensor maps (host) ----------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// Tensor map of one operand for tma_slab (extent xext along M / N, K along the reduction); false = this operand cannot
// be described (the caller takes the one-tile kernel).
template <bool KCONTIG>
bool make_operand_map(CUtensorMap* m, const float* X, long long ld, long long cblk, int xext, long long K) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || K < 32 || xext < 1 || (ld & 3) || (cblk & 3) || ((uintptr_t)X & 15)) return false;
  cuuint64_t dims[4], strides[3];
  cuuint32_t box[4], estr[4] = {1, 1, 1, 1};
  cuuint32_t rank;
  CUtensorMapSwizzle sw;
  const bool blocked = cblk != 128;
  if (KCONTIG) {                       // X[x][k]
    sw = CU_TENSOR_MAP_SWIZZLE_128B;
    if (!blocked) {
      rank = 2;
      dims[0] = (cuuint64_t)K; dims[1] = (cuuint64_t)xext;
      strides[0] = (cuuint64_t)ld * 4;
      box[0] = 32; box[1] = 128;
    } else {
      if (K & 127) return false;
      rank = 3;
      dims[0] = 128; dims[1] = (cuuint64_t)xext; dims[2] = (cuuint64_t)(K >> 7);
      strides[0] = (cuuint64_t)ld * 4; strides[1] = (cuuint64_t)cblk * 4;
      box[0] = 32; box[1] = 128; box[2] = 1;
    }
  } else {                             // X[k][x]
    sw = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    if (!blocked) {
      if (xext & 31) return false;
      rank = 3;
      dims[0] = 32; dims[1] = (cuuint64_t)K; dims[2] = (cuuint64_t)(xext >> 5);
      strides[0] = (cuuint64_t)ld * 4; strides[1] = 128;
      box[0] = 32; box[1] = 32; box[2] = 4;
    } else {
      if (xext & 127) return false;
      rank = 4;
      dims[0] = 32; dims[1] = (cuuint64_t)K; dims[2] = 4; dims[3] = (cuuint64_t)(xext >> 7);
      strides[0] = (cuuint64_t)ld * 4; strides[1] = 128; strides[2] = (cuuint64_t)cblk * 4;
      box[0] = 32; box[1] = 32; box[2] = 4; box[3] = 1;
    }
  }
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32, rank, const_cast<float*>(X), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// second stage of every split reduction: out[i] (=|+=) alpha * sum_s partial[s][i] in a FIXED order (deterministic):
// a block covers 32 consecutive outputs with LANES split lanes; lane j adds the splits j, j + LANES, ... in order (coalesced
// 128-byte reads), then the lane sums are added in lane order.  LANES = 32 for the long split lists of the column sums
// (a few outputs, hundreds of splits: a latency chain), 8 for the short ones of the split products.
template <int LANES>
__global__ void __launch_bounds__(32 * LANES)
reduce_partials_kernel(const float* __restrict__ partial, int splits, long long n, long long ldo, int ncols,
                       float alpha, int accumulate, float* __restrict__ out) {
  __shared__ float red[LANES][32];
  const int o = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * 32 + o;
  float s = 0.f;
  if (i < n) {
#pragma unroll 4
    for (int k = sl; k < splits; k += LANES) s += partial[(size_t)k * n + i];
  }
  red[sl][o] = s;
  __syncthreads();
  if (sl == 0 && i < n) {
#pragma unroll
    for (int k = 1; k < LANES; ++k) s += red[k][o];
    s *= alpha;
    float* p = out + (i / ncols) * ldo + (i % ncols);
    *p = accumulate ? *p + s : s;
  }
}

void reduce_partials(cudaStream_t s, const float* partial, int splits, long long n, long long ldo, int ncols, float alpha,
                     int accumulate, float* out) {
  const unsigned blocks = (unsigned)((n + 31) / 32);
  if (splits > 64) reduce_partials_kernel<32><<<blocks, 1024, 0, s>>>(partial, splits, n, ldo, ncols, alpha, accumulate, out);
  else reduce_partials_kernel<8><<<blocks, 256, 0, s>>>(partial, splits, n, ldo, ncols, alpha, accumulate, out);
}

struct Gemm {
  cudaStream_t s;
  float* partial;          // split-K scratch
  size_t partial_floats;
  int sms;
  bool tf32 = false;       // tensor-core TF32 products (fp32 accumulation) instead of fp32 FFMA
};

// what a launch may add to the plain product (see GemmArgs)
struct GemmOpt {
  long long a_cblk = 128, b_cblk = 128, c_cblk = 128;
  float* gelu_out = nullptr;            // C2 = gelu(C) * rowscale
  const float* gz = nullptr;            // C = (alpha A B + bias) * gelu'(gz) * rowscale
  long long gz_ld = 0;
  const float* rowscale = nullptr;      // per 16 rows of C (the cutoff window of an edge)
  const float* res_in = nullptr;        // with res_scale and gelu_out: gelu_out = res_in + res_scale[n] * C (residual update)
  const float* res_scale = nullptr;
  float* colsum_out = nullptr;          // out[n] = sum_m C[m][n] (a bias gradient) from the epilogue's own values when the
                                        // TMA kernel runs unsplit with one n tile per CTA; a separate column-sum pass otherwise
};

int colsum(const Gemm& g, const float* X, const float* Y, long long rows, int ncols, long long ld, float* out, bool accumulate);

// op: C[M,N] (=|+=) alpha A B (+bias), epilogue options in `o`.  Returns ARREAU_* / cudaError.
template <bool AK, bool BK>
int gemm(const Gemm& g, const float* A, long long lda, const float* B, long long ldb, float* C, long long ldc, int M,
         int N, long long K, float alpha, const float* bias, bool accumulate, const GemmOpt& o = GemmOpt()) {
  if (M <= 0 || N <= 0) return ARREAU_OK;
  const int tiles = ((M + kBM - 1) / kBM) * ((N + kBN - 1) / kBN);
  const bool plain_out = !bias && !o.gelu_out && !o.gz && o.c_cblk == 128 && !o.colsum_out;   // what the split second stage can finish
  // tensor maps of the operands for the TMA-fed persistent kernel; an operand it cannot describe -> one tile per CTA
  alignas(64) CUtensorMap map_a, map_b;
  const bool use_tma = g.tf32 && make_operand_map<AK>(&map_a, A, lda, o.a_cblk, M, K) &&
                       make_operand_map<BK>(&map_b, B, ldb, o.b_cblk, N, K);
  int splits = 1;
  if (K > 4096 && tiles < g.sms && plain_out) {      // reduction-dominated (weight gradients): split the rows
    splits = (2 * g.sms + tiles - 1) / tiles;
    if (use_tma) {
      // persistent kernel: items = tiles * splits should fill whole rounds of the SMs; the fewest splits that do
      // (within 3 %) keep the partial traffic and the second stage small
      double best = 0.0;
      for (int r = 1; r <= 4; ++r) {
        const int sp = r * g.sms / tiles;
        if (sp < 1) continue;
        const long long it = (long long)sp * tiles;
        const double util = (double)it / (double)(((it + g.sms - 1) / g.sms) * g.sms);
        if (util > best + 0.03) { best = util; splits = sp; }
      }
    }
    const long long max_by_k = (K + 511) / 512;
    if (splits > max_by_k) splits = (int)max_by_k;
    while (splits > 1 && (size_t)splits * M * N > g.partial_floats) --splits;
  }
  long long kps = (K + splits - 1) / splits;
  kps = (kps + 31) / 32 * 32;             // whole K slabs of both the SIMT (16) and the tcgen05 (32) kernels
  splits = (int)((K + kps - 1) / kps);
  if (splits < 1) splits = 1;
  dim3 grid((N + kBN - 1) / kBN, (M + kBM - 1) / kBM, splits);
  const int ntn = (N + kBN - 1) / kBN;
  const int ws_grid = (long long)tiles * splits < g.sms ? tiles * splits : g.sms;
  const bool fuse_colsum = o.colsum_out && use_tma && splits == 1 && ws_grid % ntn == 0 && o.c_cblk == 128 &&
                           (size_t)(ws_grid / ntn) * 4 * N <= g.partial_floats;
  GemmArgs a{A, lda, o.a_cblk, B, ldb, o.b_cblk, C, ldc, o.c_cblk, M, N, K, kps, alpha, bias, accumulate ? 1 : 0,
             g.partial, o.gelu_out, o.gz, o.gz_ld, o.rowscale, o.res_in, o.res_scale, splits,
             fuse_colsum ? g.partial : nullptr, g_ws_prof};
  if (use_tma) {
    static bool attr_set = false;       // one flag per template instance
    if (!attr_set) {
      cudaError_t e = cudaFuncSetAttribute(sgemm_tma_kernel<AK, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, wsg::kSmemBytes);
      if (e != cudaSuccess) return (int)e;
      attr_set = true;
    }
    sgemm_tma_kernel<AK, BK><<<(unsigned)ws_grid, wsg::kThreads, wsg::kSmemBytes, g.s>>>(a, map_a, map_b);
  } else if (g.tf32) {
    static bool attr_set = false;       // one flag per template instance
    if (!attr_set) {
      cudaError_t e = cudaFuncSetAttribute(sgemm_tc_kernel<AK, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, tcg::kSmemBytes);
      if (e != cudaSuccess) return (int)e;
      attr_set = true;
    }
    sgemm_tc_kernel<AK, BK><<<grid, kGT, tcg::kSmemBytes, g.s>>>(a);
  } else {
    sgemm_kernel<AK, BK><<<grid, kGT, 0, g.s>>>(a);
  }
  CUDA_LAUNCH_CHECK();
  if (splits > 1) {
    const long long n = (long long)M * N;
    reduce_partials(g.s, g.partial, splits, n, ldc, N, alpha, accumulate ? 1 : 0, C);
    CUDA_LAUNCH_CHECK();
  }
  if (fuse_colsum) {
    reduce_partials(g.s, g.partial, ws_grid / ntn * 4, N, N, N, 1.0f, 0, o.colsum_out);
    CUDA_LAUNCH_CHECK();
  } else if (o.colsum_out) {
    return colsum(g, C, nullptr, M, N, ldc, o.colsum_out, false);
  }
  return ARREAU_OK;
}

// ================================================================================================
// column sums over rows (bias / scale gradients): out[c] (=|+=) sum_r X[r][c] (* Y[r][c])
// two stages, fixed order.  ncols % 128 == 0.
// ================================================================================================
constexpr int kColSplits = 592;     // 4 blocks of 256 threads per SM

template <bool PROD>
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ X, const float* __restrict__ Y, long long rows, int ncols, long long ld,
              float* __restrict__ partial) {
  // block = 256 threads = (256 / (ncols / 4)) row lanes x (ncols / 4) float4 columns; blockIdx.x = row split.  Each
  // thread keeps 4 independent 16-byte loads in flight; the row lanes are combined in shared memory in a fixed order.
  __shared__ float4 red[256];
  const int c4n = ncols >> 2, lanes = 256 / c4n;
  const int c4 = threadIdx.x % c4n, rl = threadIdx.x / c4n;
  const long long per = (rows + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f), s1 = s0, s2 = s0, s3 = s0;
  auto ld4 = [&](long long r) {
    float4 a = __ldg(reinterpret_cast<const float4*>(X + r * ld) + c4);
    if (PROD) {
      const float4 y = __ldg(reinterpret_cast<const float4*>(Y + r * ld) + c4);
      a.x *= y.x; a.y *= y.y; a.z *= y.z; a.w *= y.w;
    }
    return a;
  };
  auto acc = [](float4& s, const float4& a) { s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w; };
  long long r = r0 + rl;
  for (; r + 3LL * lanes < r1; r += 4LL * lanes) {
    const float4 a0 = ld4(r), a1 = ld4(r + lanes), a2 = ld4(r + 2LL * lanes), a3 = ld4(r + 3LL * lanes);
    acc(s0, a0); acc(s1, a1); acc(s2, a2); acc(s3, a3);
  }
  for (; r < r1; r += lanes) acc(s0, ld4(r));
  acc(s0, s1); acc(s2, s3); acc(s0, s2);
  red[threadIdx.x] = s0;
  __syncthreads();
  if (rl == 0) {
    for (int k = 1; k < lanes; ++k) acc(s0, red[k * c4n + c4]);          // fixed order: deterministic
    reinterpret_cast<float4*>(partial + (size_t)blockIdx.x * ncols)[c4] = s0;
  }
}

int colsum(const Gemm& g, const float* X, const float* Y, long long rows, int ncols, long long ld, float* out,
           bool accumulate) {
  if (ncols % 128 != 0 || ncols > 1024 || ld % 4 != 0) return ARREAU_ERR_UNSUPPORTED;
  if (rows <= 0) return ARREAU_OK;
  // enough row splits to put ~2 blocks on every SM, at least 64 rows each, bounded by the split scratch
  long long splits = (rows + 63) / 64;
  if (splits > kColSplits) splits = kColSplits;
  while (splits > 1 && (size_t)splits * ncols > g.partial_floats) --splits;
  if (Y) colsum_kernel<true><<<(unsigned)splits, 256, 0, g.s>>>(X, Y, rows, ncols, ld, g.partial);
  else colsum_kernel<false><<<(unsigned)splits, 256, 0, g.s>>>(X, nullptr, rows, ncols, ld, g.partial);
  CUDA_LAUNCH_CHECK();
  reduce_partials(g.s, g.partial, (int)splits, ncols, ncols, ncols, 1.0f, accumulate ? 1 : 0, out);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

// ================================================================================================
// elementwise / rowwise kernels
// ================================================================================================
// a = gelu(z) [* rowscale[r / rows_per_scale]]
__global__ void gelu_fwd_kernel(const float* __restrict__ z, long long n, int ncols, const float* __restrict__ rowscale,
                                int rows_per_scale, float* __restrict__ a) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  const float4 v = *reinterpret_cast<const float4*>(z + i);
  const float sc = rowscale ? rowscale[(i / ncols) / rows_per_scale] : 1.0f;
  *reinterpret_cast<float4*>(a + i) = make_float4(gelu_erf(v.x) * sc, gelu_erf(v.y) * sc, gelu_erf(v.z) * sc, gelu_erf(v.w) * sc);
}

// dz = da * gelu'(z) [* rowscale]      (in place on da allowed)
__global__ void gelu_bwd_kernel(const float* __restrict__ z, const float* da, long long n, int ncols,
                                const float* __restrict__ rowscale, int rows_per_scale, float* dz) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  const float4 v = *reinterpret_cast<const float4*>(z + i);
  const float4 d = *reinterpret_cast<const float4*>(da + i);
  const float sc = rowscale ? rowscale[(i / ncols) / rows_per_scale] : 1.0f;
  *reinterpret_cast<float4*>(dz + i) = make_float4(d.x * gelu_grad(v.x) * sc, d.y * gelu_grad(v.y) * sc,
                                                   d.z * gelu_grad(v.z) * sc, d.w * gelu_grad(v.w) * sc);
}

// Backward of the residual update h_out = h_in + ls * m (convnext.py:31-32) in one pass over dh and m:
//   dm = dh * ls (written), partial[block] = [ sum_r dh * m  (d layer_scale) | sum_r dm  (d lin2 bias) ]
// block = 256 threads = 8 row lanes x 32 float4 columns, blockIdx.x = row split; fixed-order combination (deterministic).
__global__ void __launch_bounds__(256)
ls_bwd_kernel(const float* __restrict__ dh, const float* __restrict__ m, const float* __restrict__ ls, long long rows,
              float* __restrict__ dm, float* __restrict__ partial) {
  __shared__ float4 red[2][256];
  const int c4 = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const long long per = (rows + gridDim.x - 1) / gridDim.x;
  const long long r0 = (long long)blockIdx.x * per, r1 = (r0 + per < rows) ? r0 + per : rows;
  const float4 sc = reinterpret_cast<const float4*>(ls)[c4];
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
#pragma unroll 4
  for (long long r = r0 + rl; r < r1; r += 8) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(dh + r * kC) + c4);
    const float4 mv = __ldg(reinterpret_cast<const float4*>(m + r * kC) + c4);
    const float4 d = make_float4(g.x * sc.x, g.y * sc.y, g.z * sc.z, g.w * sc.w);
    reinterpret_cast<float4*>(dm + r * kC)[c4] = d;
    s1.x = fmaf(g.x, mv.x, s1.x); s1.y = fmaf(g.y, mv.y, s1.y); s1.z = fmaf(g.z, mv.z, s1.z); s1.w = fmaf(g.w, mv.w, s1.w);
    s2.x += d.x; s2.y += d.y; s2.z += d.z; s2.w += d.w;
  }
  red[0][threadIdx.x] = s1;
  red[1][threadIdx.x] = s2;
  __syncthreads();
  if (rl < 2) {                              // row lane 0 finishes the first sum, row lane 1 the second
    float4 a = red[rl][c4];
    for (int k = 1; k < 8; ++k) {
      const float4 v = red[rl][k * 32 + c4];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    reinterpret_cast<float4*>(partial + (size_t)blockIdx.x * 2 * kC + rl * kC)[c4] = a;
  }
}

__global__ void fill_kernel(float* __restrict__ p, long long n, float v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// ---- edge rows: invariants -> 83 monomials (+ constant 1, zero padding to 128) and the cutoff window ----------
// (geometry/invariants.py:17-22, transforms/invariants.py:81-87, embedding.py:10-14, windowing.py:21-29)
// A block takes 64 (edge, orientation) rows: one thread per row forms its monomials in shared memory, then the whole block
// writes the 64 x 128 tile with coalesced 16-byte stores (one thread per row writing its own 512-byte row straight to
// global memory took 242 us for the C5 batch's 146 MB; this form is HBM-bound).
constexpr int kMonoRows = 64;
__global__ void __launch_bounds__(128)
edge_mono_kernel(const double* __restrict__ dir, const double* __restrict__ dist, const double* __restrict__ lattice,
                 const int32_t* __restrict__ crystal_of_atom, const int32_t* __restrict__ src,
                 const int32_t* __restrict__ num_edges_ptr, long long edge_capacity, const float* __restrict__ ori,
                 double radius, float* __restrict__ mono, float* __restrict__ win) {
  __shared__ float tile[kMonoRows][129];
  const long long row0 = (long long)blockIdx.x * kMonoRows, total = edge_capacity * kO;
  long long E = *num_edges_ptr;
  if (E > edge_capacity) E = edge_capacity;
  const int t = threadIdx.x;
  if (t < kMonoRows && row0 + t < total) {
    const long long row = row0 + t, e = row >> 4;
    const int o = (int)(row & (kO - 1));
    float* out = tile[t];
    if (e >= E) {
      for (int k = 0; k <= kMono; ++k) out[k] = 0.f;
      if (o == 0) win[e] = 0.f;
    } else {
      float attr[6];
      edge_invariants(dir + 3 * e, dist[e], lattice + 9 * (size_t)crystal_of_atom[src[e]], ori + 3 * o, attr);
      monomials83(attr, out, 1);
      out[kMono] = 1.0f;
      if (o == 0) win[e] = cutoff_window(dist[e], radius);
    }
  }
  __syncthreads();
  for (int i = t; i < kMonoRows * 32; i += 128) {
    const int r = i >> 5, c = (i & 31) * 4;
    if (row0 + r >= total) break;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c <= kMono) v = make_float4(tile[r][c], tile[r][c + 1], tile[r][c + 2], tile[r][c + 3]);   // kMono + 1 = 84 = 21 * 4
    *reinterpret_cast<float4*>(mono + (row0 + r) * 128 + c) = v;
  }
}

// ---- LayerNorm over C = 128 channels, one warp per row (convnext.py:25) -------------------------------------
__global__ void __launch_bounds__(256)
ln_fwd_kernel(const float* __restrict__ x2, const float* __restrict__ gw, const float* __restrict__ gb, long long rows,
              float* __restrict__ y) {
  const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float4 t = *reinterpret_cast<const float4*>(x2 + r * kC + lane * 4);
  const float mean = warp_sum((t.x + t.y) + (t.z + t.w)) * (1.0f / kC);
  const float dx = t.x - mean, dy = t.y - mean, dz = t.z - mean, dw = t.w - mean;
  const float var = warp_sum((dx * dx + dy * dy) + (dz * dz + dw * dw)) * (1.0f / kC);
  const float rstd = 1.0f / sqrtf(var + 1e-5f);
  const float4 w = *reinterpret_cast<const float4*>(gw + lane * 4), b = *reinterpret_cast<const float4*>(gb + lane * 4);
  *reinterpret_cast<float4*>(y + r * kC + lane * 4) =
      make_float4(dx * rstd * w.x + b.x, dy * rstd * w.y + b.y, dz * rstd * w.z + b.z, dw * rstd * w.w + b.w);
}

// dx2 = rstd (g - mean(g) - xhat mean(g xhat)), g = dy * gamma; per-block partials of
// dgamma = sum dy xhat, dbeta = sum dy, dbias(conv) = sum dx2    -> partial[block][3][128]
constexpr int kLnWarps = 8;
__global__ void __launch_bounds__(kLnWarps * 32)
ln_bwd_kernel(const float* __restrict__ x2, const float* __restrict__ dy, const float* __restrict__ gw, long long rows,
              float* __restrict__ dx2, float* __restrict__ partial) {
  __shared__ float red[kLnWarps][3][kC];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float4 w = *reinterpret_cast<const float4*>(gw + lane * 4);
  float4 sg = make_float4(0.f, 0.f, 0.f, 0.f), sb = sg, sx = sg;
  for (long long r = (long long)blockIdx.x * kLnWarps + warp; r < rows; r += (long long)gridDim.x * kLnWarps) {
    const float4 t = *reinterpret_cast<const float4*>(x2 + r * kC + lane * 4);
    const float4 d = *reinterpret_cast<const float4*>(dy + r * kC + lane * 4);
    const float mean = warp_sum((t.x + t.y) + (t.z + t.w)) * (1.0f / kC);
    const float cx = t.x - mean, cy = t.y - mean, cz = t.z - mean, cw = t.w - mean;
    const float var = warp_sum((cx * cx + cy * cy) + (cz * cz + cw * cw)) * (1.0f / kC);
    const float rstd = 1.0f / sqrtf(var + 1e-5f);
    const float hx = cx * rstd, hy = cy * rstd, hz = cz * rstd, hw = cw * rstd;
    const float gx = d.x * w.x, gy = d.y * w.y, gz = d.z * w.z, gw_ = d.w * w.w;
    const float m1 = warp_sum((gx + gy) + (gz + gw_)) * (1.0f / kC);
    const float m2 = warp_sum((gx * hx + gy * hy) + (gz * hz + gw_ * hw)) * (1.0f / kC);
    const float4 o = make_float4(rstd * (gx - m1 - hx * m2), rstd * (gy - m1 - hy * m2), rstd * (gz - m1 - hz * m2),
                                 rstd * (gw_ - m1 - hw * m2));
    *reinterpret_cast<float4*>(dx2 + r * kC + lane * 4) = o;
    sg.x += d.x * hx; sg.y += d.y * hy; sg.z += d.z * hz; sg.w += d.w * hw;
    sb.x += d.x; sb.y += d.y; sb.z += d.z; sb.w += d.w;
    sx.x += o.x; sx.y += o.y; sx.z += o.z; sx.w += o.w;
  }
  *reinterpret_cast<float4*>(&red[warp][0][lane * 4]) = sg;
  *reinterpret_cast<float4*>(&red[warp][1][lane * 4]) = sb;
  *reinterpret_cast<float4*>(&red[warp][2][lane * 4]) = sx;
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * kC; i += blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < kLnWarps; ++k) s += red[k][i / kC][i % kC];
    partial[(size_t)blockIdx.x * 3 * kC + i] = s;
  }
}

// ---- fiber conv backward (conv.py:115): x2[b,p,c] = (1/O) sum_o x1[b,o,c] fk[o,p,c] ------------------------
// dx1[b,o,c] = (1/O) sum_p dx2[b,p,c] fk[o,p,c]; block = kDx1Atoms atoms, thread = channel (every fiber-kernel value read
// from L1 serves all of them; N / kDx1Atoms independent blocks instead of 2 per SM looping over their atoms)
constexpr int kDx1Atoms = 4;
__global__ void __launch_bounds__(kC)
fiber_bwd_dx1_kernel(const float* __restrict__ dx2, const float* __restrict__ fk, int N, float* __restrict__ dx1) {
  const int c = threadIdx.x;
  const int b0 = kDx1Atoms * blockIdx.x;
  float d[kDx1Atoms][kO];
#pragma unroll
  for (int a = 0; a < kDx1Atoms; ++a) {
    const int b = b0 + a < N ? b0 + a : N - 1;
#pragma unroll
    for (int p = 0; p < kO; ++p) d[a][p] = dx2[((size_t)b * kO + p) * kC + c];
  }
#pragma unroll 2
  for (int o = 0; o < kO; ++o) {
    float s[kDx1Atoms];
#pragma unroll
    for (int a = 0; a < kDx1Atoms; ++a) s[a] = 0.f;
#pragma unroll
    for (int p = 0; p < kO; ++p) {
      const float f = __ldg(fk + ((size_t)o * kO + p) * kC + c);
#pragma unroll
      for (int a = 0; a < kDx1Atoms; ++a) s[a] = fmaf(d[a][p], f, s[a]);
    }
#pragma unroll
    for (int a = 0; a < kDx1Atoms; ++a)
      if (b0 + a < N) dx1[((size_t)(b0 + a) * kO + o) * kC + c] = s[a] * (1.0f / kO);
  }
}

// dfk[o,p,c] = (1/O) sum_b x1[b,o,c] dx2[b,p,c]: 1024 threads = (o pair, channel), atoms strided over blocks,
// per-block partial [O][O][C]
__global__ void __launch_bounds__(1024)
fiber_bwd_dfk_kernel(const float* __restrict__ x1, const float* __restrict__ dx2, int N, float* __restrict__ partial) {
  const int c = threadIdx.x & (kC - 1), og = threadIdx.x >> 7;   // og in 0..7 -> o = 2 og, 2 og + 1
  float acc[2][kO];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int p = 0; p < kO; ++p) acc[i][p] = 0.f;
  for (int b = blockIdx.x; b < N; b += gridDim.x) {
    const float xa = x1[((size_t)b * kO + 2 * og) * kC + c], xb = x1[((size_t)b * kO + 2 * og + 1) * kC + c];
#pragma unroll
    for (int p = 0; p < kO; ++p) {
      const float d = dx2[((size_t)b * kO + p) * kC + c];
      acc[0][p] = fmaf(xa, d, acc[0][p]);
      acc[1][p] = fmaf(xb, d, acc[1][p]);
    }
  }
  float* out = partial + (size_t)blockIdx.x * kO * kO * kC;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int p = 0; p < kO; ++p) out[((size_t)(2 * og + i) * kO + p) * kC + c] = acc[i][p];
}

// ---- message pass backward (conv.py:131-133 + PyG add aggregation) -------------------------------------------
// dh[j,o,c] += sum_{e: src_e = j} kern[e,o,c] * dx1[dst_e,o,c]   (edges of j's crystal scanned in edge order:
// deterministic, no atomics) and, in the same pass over j's outgoing edges, their rows of the kernel gradient
// dkern[e,o,c] = dx1[dst_e,o,c] * h[j,o,c] (every edge has exactly one sender, so every row is written exactly once and
// dx1[dst_e] is fetched once for both).  One block per sender atom; a thread owns 8 of the 2048 (o,c) entries.  The blocks
// beyond the atoms zero the rows of the unused edge capacity (the weight-gradient product reduces over all of it).
constexpr int kDkernTailBlocks = 32;
__global__ void __launch_bounds__(256)
message_bwd_kernel(const float* __restrict__ kern, const float* __restrict__ dx1, const float* __restrict__ h,
                   const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                   const int32_t* __restrict__ atom_offset, const int32_t* __restrict__ crystal_of_atom,
                   const int32_t* __restrict__ num_edges_ptr, long long edge_capacity, int N, float* __restrict__ dh,
                   float* __restrict__ dkern) {
  __shared__ int s_list[256];
  __shared__ int s_wcount[8];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if ((int)blockIdx.x >= N) {
    long long E = *num_edges_ptr;
    if (E > edge_capacity) E = edge_capacity;
    const long long lo = E * (kO * kC / 4), hi = edge_capacity * (kO * kC / 4);
    for (long long i = lo + (long long)(blockIdx.x - N) * 256 + tid; i < hi; i += (long long)kDkernTailBlocks * 256)
      reinterpret_cast<float4*>(dkern)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    return;
  }
  const int j = blockIdx.x;
  const int g = crystal_of_atom[j];
  long long e_lo = row_ptr[atom_offset[g]], e_hi = row_ptr[atom_offset[g + 1]];
  if (e_hi > edge_capacity) e_hi = edge_capacity;
  float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
  const int i0 = tid * 4, i1 = 1024 + tid * 4;
  const float4 h0 = *reinterpret_cast<const float4*>(h + (size_t)j * kO * kC + i0);
  const float4 h1 = *reinterpret_cast<const float4*>(h + (size_t)j * kO * kC + i1);
  for (long long base = e_lo; base < e_hi; base += 256) {
    const long long e = base + tid;
    const bool match = e < e_hi && src[e] == j;
    const unsigned bal = __ballot_sync(0xffffffffu, match);
    if (lane == 0) s_wcount[warp] = __popc(bal);
    __syncthreads();
    int off = 0, total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      if (w < warp) off += s_wcount[w];
      total += s_wcount[w];
    }
    if (match) s_list[off + __popc(bal & ((1u << lane) - 1u))] = (int)(e - base);
    __syncthreads();
#pragma unroll 2
    for (int m = 0; m < total; ++m) {
      const long long ee = base + s_list[m];
      const size_t ko = (size_t)ee * kO * kC, xo = (size_t)dst[ee] * kO * kC;
      const float4 k0 = *reinterpret_cast<const float4*>(kern + ko + i0), k1 = *reinterpret_cast<const float4*>(kern + ko + i1);
      const float4 d0 = *reinterpret_cast<const float4*>(dx1 + xo + i0), d1 = *reinterpret_cast<const float4*>(dx1 + xo + i1);
      acc0.x = fmaf(k0.x, d0.x, acc0.x); acc0.y = fmaf(k0.y, d0.y, acc0.y);
      acc0.z = fmaf(k0.z, d0.z, acc0.z); acc0.w = fmaf(k0.w, d0.w, acc0.w);
      acc1.x = fmaf(k1.x, d1.x, acc1.x); acc1.y = fmaf(k1.y, d1.y, acc1.y);
      acc1.z = fmaf(k1.z, d1.z, acc1.z); acc1.w = fmaf(k1.w, d1.w, acc1.w);
      *reinterpret_cast<float4*>(dkern + ko + i0) = make_float4(d0.x * h0.x, d0.y * h0.y, d0.z * h0.z, d0.w * h0.w);
      *reinterpret_cast<float4*>(dkern + ko + i1) = make_float4(d1.x * h1.x, d1.y * h1.y, d1.z * h1.z, d1.w * h1.w);
    }
    __syncthreads();
  }
  float* p = dh + (size_t)j * kO * kC;
  float4 a = *reinterpret_cast<float4*>(p + i0), b = *reinterpret_cast<float4*>(p + i1);
  a.x += acc0.x; a.y += acc0.y; a.z += acc0.z; a.w += acc0.w;
  b.x += acc1.x; b.y += acc1.y; b.z += acc1.z; b.w += acc1.w;
  *reinterpret_cast<float4*>(p + i0) = a;
  *reinterpret_cast<float4*>(p + i1) = b;
}

// ---- read-out gradient rows (ponita.py:105-117,152; to_from_sphere.py:10-14) ---------------------------------
// dr[(b,o)][z] for the per-orientation read-out r_l[b,o,:] of ANY layer (the layers are averaged):
//   z < Z: dlogits[b,z] / (L O);  z == Z: sum_d dscore[b,d] ori[o,d] / (L O);  Z < z < Z+4: dlen0[g(b), z-Z-1] / (L O)
//   columns Z+4 .. 127 are zero padding.
__global__ void __launch_bounds__(128)
readout_grad_rows_kernel(const float* __restrict__ dlogits, const float* __restrict__ dscore,
                         const float* __restrict__ dlen0, const int32_t* __restrict__ crystal_of_atom,
                         const float* __restrict__ ori, int N, int Z, float scale, float* __restrict__ dr) {
  const long long row = blockIdx.x;
  const int b = (int)(row >> 4), o = (int)(row & (kO - 1)), z = threadIdx.x;
  if (b >= N) return;
  float v = 0.f;
  if (z < Z) v = dlogits[(size_t)b * Z + z];
  else if (z == Z) v = dscore[3 * b] * ori[3 * o] + dscore[3 * b + 1] * ori[3 * o + 1] + dscore[3 * b + 2] * ori[3 * o + 2];
  else if (z < Z + 4) v = dlen0[3 * crystal_of_atom[b] + (z - Z - 1)];
  dr[row * 128 + z] = v * scale;
}

// x_lift[(b,o)][0..F) = x[b], [F..F+V) = vec[b,v] . ori[o], zero padded to `pitch` (position_orientation_graph.py:84-86)
__global__ void __launch_bounds__(256)
lift_rows_kernel(const float* __restrict__ x, const float* __restrict__ vec, const float* __restrict__ ori, int N, int F,
                 int V, int pitch, float* __restrict__ xl) {
  const long long row = blockIdx.x;
  const int b = (int)(row >> 4), o = (int)(row & (kO - 1));
  if (b >= N) return;
  for (int f = threadIdx.x; f < pitch; f += blockDim.x) {
    float v = 0.f;
    if (f < F) v = x[(size_t)b * F + f];
    else if (f < F + V) {
      const float* p = vec + ((size_t)b * V + (f - F)) * 3;
      v = p[0] * ori[3 * o] + p[1] * ori[3 * o + 1] + p[2] * ori[3 * o + 2];
    }
    xl[row * pitch + f] = v;
  }
}

// fiber rows: [fa, fa^2, fa^3, 1, 0...] (16 wide), fa = ori_o . ori_p   (geometry/invariants.py:23, embedding.py)
__global__ void fiber_rows_kernel(const float* __restrict__ ori, float* __restrict__ rows16) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= kO * kO) return;
  const int o = r / kO, p = r % kO;
  const float fa = ori[3 * o] * ori[3 * p] + ori[3 * o + 1] * ori[3 * p + 1] + ori[3 * o + 2] * ori[3 * p + 2];
  float* out = rows16 + r * 16;
  out[0] = fa; out[1] = fa * fa; out[2] = fa * fa * fa; out[3] = 1.0f;
  for (int k = 4; k < 16; ++k) out[k] = 0.f;
}

// folded first basis layer W1m[c][0..82] = sum of basis_fn.1.weight columns of equal monomials, [83] = bias, rest 0
// (pitch 128), and the gradient scatter back: dW1[c][f] = dW1m[c][fold[f]], db1[c] = dW1m[c][83]
__global__ void fold_w1_kernel(const float* __restrict__ w1, const float* __restrict__ b1, const int32_t* __restrict__ fold,
                               int nfeat, float* __restrict__ w1m) {
  const int c = blockIdx.x, k = threadIdx.x;   // 128 threads
  float s = 0.f;
  if (k < kMono) {
    for (int f = 0; f < nfeat; ++f)
      if (fold[f] == k) s += w1[(size_t)c * nfeat + f];
  } else if (k == kMono) {
    s = b1[c];
  }
  w1m[c * 128 + k] = s;
}
// the same fold in the forward's layout: w1m_t[k][c], k < 96 (rows 84..95 zero)
__global__ void fold_w1_t_kernel(const float* __restrict__ w1, const float* __restrict__ b1, const int32_t* __restrict__ fold,
                                 int nfeat, float* __restrict__ w1m_t) {
  const int k = blockIdx.x, c = threadIdx.x;   // grid 96, 128 threads
  float s = 0.f;
  if (k < kMono) {
    for (int f = 0; f < nfeat; ++f)
      if (fold[f] == k) s += w1[(size_t)c * nfeat + f];
  } else if (k == kMono) {
    s = b1[c];
  }
  w1m_t[k * kC + c] = s;
}
__global__ void unfold_w1_grad_kernel(const float* __restrict__ dw1m, const int32_t* __restrict__ fold, int nfeat,
                                      float* __restrict__ dw1, float* __restrict__ db1) {
  const int c = blockIdx.x;
  for (int f = threadIdx.x; f < nfeat; f += blockDim.x) dw1[(size_t)c * nfeat + f] = dw1m[c * 128 + fold[f]];
  if (threadIdx.x == 0) db1[c] = dw1m[c * 128 + kMono];
}
// fiber first layer: W1f16[c][0..2] = fiber_basis_fn.1.weight[c], [3] = bias, rest 0 (pitch 16) and back
__global__ void pack_fiber_w1_kernel(const float* __restrict__ w1, const float* __restrict__ b1, float* __restrict__ w16) {
  const int c = blockIdx.x, k = threadIdx.x;   // 16 threads
  w16[c * 16 + k] = k < 3 ? w1[c * 3 + k] : (k == 3 ? b1[c] : 0.f);
}
__global__ void unpack_fiber_w1_grad_kernel(const float* __restrict__ d16, float* __restrict__ dw1, float* __restrict__ db1) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= kC) return;
  dw1[c * 3] = d16[c * 16]; dw1[c * 3 + 1] = d16[c * 16 + 1]; dw1[c * 3 + 2] = d16[c * 16 + 2];
  db1[c] = d16[c * 16 + 3];
}

// sum and sum of squares of a tensor in fp64 (std for FiberBundleConv.callibrate, conv.py:122-123): two stages
__global__ void __launch_bounds__(256)
moments_kernel(const float* __restrict__ x, const float* __restrict__ sub_cols, long long n, double* __restrict__ partial) {
  __shared__ double sh[2][8];
  double s = 0.0, q = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double v = (double)x[i];
    if (sub_cols) v -= (double)sub_cols[i & (kC - 1)];
    s += v;
    q += v * v;
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = s; sh[1][threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, tq = 0.0;
    for (int k = 0; k < 8; ++k) { ts += sh[0][k]; tq += sh[1][k]; }
    partial[2 * blockIdx.x] = ts;
    partial[2 * blockIdx.x + 1] = tq;
  }
}
// one warp: lane l adds the blocks l, l + 32, ... in order, then a fixed shuffle tree (deterministic; one thread walking all
// the partials was a 16 us chain of dependent loads once per training step)
__global__ void moments_finish_kernel(const double* __restrict__ partial, int blocks, double* __restrict__ out) {
  if (blockIdx.x != 0 || threadIdx.x >= 32) return;
  double s = 0.0, q = 0.0;
  for (int k = threadIdx.x; k < blocks; k += 32) { s += partial[2 * k]; q += partial[2 * k + 1]; }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, off);
    q += __shfl_xor_sync(0xffffffffu, q, off);
  }
  if (threadIdx.x == 0) {
    out[0] = s;
    out[1] = q;
  }
}

int sm_count() {
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
  }
  return sms;
}

inline unsigned blocks_for(long long n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }

#define TRY(call)                          \
  do {                                     \
    const int rc__ = (call);               \
    if (rc__ != ARREAU_OK) return rc__;    \
  } while (0)

// carve a float workspace
struct Carver {
  float* base;
  size_t used = 0;
  explicit Carver(float* b) : base(b) {}
  float* take(size_t n) {
    float* p = base ? base + used : nullptr;
    used += (n + 63) & ~(size_t)63;      // 256-byte granules
    return p;
  }
};

constexpr size_t kPartialFloats = (size_t)8 << 20;   // 32 MB of split scratch
constexpr int kDfkBlocks = 148;
constexpr int kLnBlocks = 296;

struct BwdBuffers {
  // edge rows (Re = edge_capacity * O)
  float *mono, *z1, *a1, *z2, *kb, *dkb, *dkern, *da1, *win;   // dkern: [L][Re][C], the gradient slabs of every layer
  // node rows (Rn = N * O)
  float *dh, *dr, *y, *z, *a, *m, *dm, *da, *dy, *dx2, *dx1, *xl;
  // fiber chain (256 rows)
  float *frow, *fz1, *fa1, *fz2, *fkb, *dfk, *dfkb, *fda1, *fw16, *fdw16;
  float *w1m, *dw1m, *partial, *small;   // small: [128 x 640] scratch for narrow outputs
  // kept by arreau_ponita_forward_train, one slab per layer: LayerNorm output y [Rn][C], ConvNext hidden pre-activation
  // z [Rn][W], its GELU a [Rn][W], the MLP output m [Rn][C]
  float *ys, *zs, *as, *ms;
  size_t total;
};

BwdBuffers carve(float* base, long long N, long long Ecap, int xl_pitch) {
  Carver c(base);
  BwdBuffers b;
  const size_t Re = (size_t)Ecap * kO, Rn = (size_t)N * kO;
  b.mono = c.take(Re * 128); b.z1 = c.take(Re * kC); b.a1 = c.take(Re * kC); b.z2 = c.take(Re * kD);
  b.kb = c.take(Re * kD); b.dkb = c.take(Re * kD); b.dkern = c.take((size_t)kL * Re * kC); b.da1 = c.take(Re * kC);
  b.win = c.take((size_t)Ecap);
  b.dh = c.take(Rn * kC); b.dr = c.take(Rn * 128); b.y = c.take(Rn * kC); b.z = c.take(Rn * kW); b.a = c.take(Rn * kW);
  b.m = c.take(Rn * kC); b.dm = c.take(Rn * kC); b.da = c.take(Rn * kW); b.dy = c.take(Rn * kC); b.dx2 = c.take(Rn * kC);
  b.dx1 = c.take(Rn * kC); b.xl = c.take(Rn * xl_pitch);
  const size_t Rf = kO * kO;
  b.frow = c.take(Rf * 16); b.fz1 = c.take(Rf * kC); b.fa1 = c.take(Rf * kC); b.fz2 = c.take(Rf * kD);
  b.fkb = c.take(Rf * kD); b.dfk = c.take((size_t)kL * Rf * kC); b.dfkb = c.take(Rf * kD); b.fda1 = c.take(Rf * kC);
  b.fw16 = c.take(kC * 16); b.fdw16 = c.take(kC * 16);
  b.w1m = c.take(kC * 128); b.dw1m = c.take(kC * 128);
  b.partial = c.take(kPartialFloats);
  b.small = c.take((size_t)128 * kL * kC);
  b.ys = c.take((size_t)kL * Rn * kC); b.zs = c.take((size_t)kL * Rn * kW); b.as = c.take((size_t)kL * Rn * kW);
  b.ms = c.take((size_t)kL * Rn * kC);
  b.total = c.used;
  return b;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
// Edge chain forward: monomials -> z1 -> a1 = gelu(z1) -> z2 -> kb = gelu(z2) * window, every matrix kept in the
// workspace for the backward (geometry/invariants.py:10-31, embedding.py:10-14, ponita.py:65,94, windowing.py:21-29).
// The activations leave the GEMMs' epilogues next to their pre-activations (no element-wise pass in between).
static int edge_chain_forward(const Gemm& g, const BwdBuffers& b, const float* P, const arreau_train_layout_t* lay,
                              const arreau_weights* w, const int32_t* fold_table, const int32_t* src, const double* dist,
                              const double* dir, const double* lattice, const int32_t* crystal_of_atom,
                              const int32_t* num_edges_ptr, long long Ecap, double radius) {
  cudaStream_t s = g.s;
  const long long Re = Ecap * kO;
  fold_w1_kernel<<<kC, 128, 0, s>>>(P + lay->basis_w1, P + lay->basis_b1, fold_table, 258, b.w1m);
  CUDA_LAUNCH_CHECK();
  if (Re <= 0) return ARREAU_OK;
  edge_mono_kernel<<<blocks_for(Re, kMonoRows), 128, 0, s>>>(dir, dist, lattice, crystal_of_atom, src, num_edges_ptr, Ecap,
                                                             w->ori, radius, b.mono, b.win);
  CUDA_LAUNCH_CHECK();
  GemmOpt o1;
  o1.gelu_out = b.a1;
  TRY((gemm<true, true>(g, b.mono, 128, b.w1m, 128, b.z1, kC, (int)Re, kC, kMonoPad, 1.f, nullptr, false, o1)));
  GemmOpt o2;
  o2.gelu_out = b.kb;
  o2.rowscale = b.win;
  TRY((gemm<true, true>(g, b.a1, kC, P + lay->basis_w2, kC, b.z2, kD, (int)Re, kD, kC, 1.f, P + lay->basis_b2, false, o2)));
  return ARREAU_OK;
}

// Fiber chain forward (geometry/invariants.py:23, ponita.py:66,95): rows (o, p) -> [fa, fa^2, fa^3, 1] -> fz1 -> fa1 -> fz2 ->
// fkb, kept for the backward; with `fiber_kernel` the five fiber kernels fkb Wf_l^T (conv.py:113) as ONE product whose
// output columns are the per-layer [O*O][C] slabs.
static int fiber_chain_forward(const Gemm& g, const BwdBuffers& b, const float* P, const arreau_train_layout_t* lay,
                               const float* ori, float* fiber_kernel) {
  cudaStream_t s = g.s;
  const int Rf = kO * kO;
  fiber_rows_kernel<<<1, 256, 0, s>>>(ori, b.frow);
  CUDA_LAUNCH_CHECK();
  pack_fiber_w1_kernel<<<kC, 16, 0, s>>>(P + lay->fiber_w1, P + lay->fiber_b1, b.fw16);
  CUDA_LAUNCH_CHECK();
  GemmOpt o1;
  o1.gelu_out = b.fa1;
  TRY((gemm<true, true>(g, b.frow, 16, b.fw16, 16, b.fz1, kC, Rf, kC, 16, 1.f, nullptr, false, o1)));
  GemmOpt o2;
  o2.gelu_out = b.fkb;
  TRY((gemm<true, true>(g, b.fa1, kC, P + lay->fiber_w2, kC, b.fz2, kD, Rf, kD, kC, 1.f, P + lay->fiber_b2, false, o2)));
  if (fiber_kernel) {
    GemmOpt o3;
    o3.c_cblk = (long long)Rf * kC;
    TRY((gemm<true, true>(g, b.fkb, kD, P + lay->conv_fiber_w, kD, fiber_kernel, kC, Rf, kL * kC, kD, 1.f, nullptr, false, o3)));
  }
  return ARREAU_OK;
}

extern "C" int arreau_train_layout(int32_t num_scalar, int32_t num_vec, int32_t num_states, arreau_train_layout_t* lay) {
  if (!lay) return ARREAU_ERR_NULL;
  if (num_scalar <= 0 || num_vec < 0 || num_states <= 0) return ARREAU_ERR_BAD_SHAPE;
  const int64_t R = num_states + 4, FV = num_scalar + num_vec;
  int64_t o = 0;
  auto put = [&](int64_t& field, int64_t n) { field = o; o += n; };
  put(lay->basis_w1, (int64_t)kC * 258); put(lay->basis_b1, kC); put(lay->basis_w2, (int64_t)kD * kC); put(lay->basis_b2, kD);
  put(lay->fiber_w1, kC * 3); put(lay->fiber_b1, kC); put(lay->fiber_w2, (int64_t)kD * kC); put(lay->fiber_b2, kD);
  put(lay->embed_w, kC * FV);
  put(lay->layer_scale, kL * kC); put(lay->conv_bias, kL * kC); put(lay->conv_kernel_w, (int64_t)kL * kC * kD);
  put(lay->conv_fiber_w, (int64_t)kL * kC * kD); put(lay->lin1_w, (int64_t)kL * kW * kC); put(lay->lin1_b, kL * kW);
  put(lay->lin2_w, (int64_t)kL * kC * kW); put(lay->lin2_b, kL * kC); put(lay->norm_w, kL * kC); put(lay->norm_b, kL * kC);
  put(lay->readout_w, kL * R * kC); put(lay->readout_b, kL * R);
  lay->total = o;
  return ARREAU_OK;
}

extern "C" int64_t arreau_ponita_backward_workspace_bytes(int32_t N, int64_t edge_capacity, int32_t num_scalar,
                                                          int32_t num_vec) {
  if (N < 0 || edge_capacity < 0) return ARREAU_ERR_BAD_SHAPE;
  const int xl_pitch = ((num_scalar + num_vec + 127) / 128) * 128;
  return (int64_t)(carve(nullptr, N, edge_capacity, xl_pitch).total * sizeof(float));
}

extern "C" int arreau_fold_basis_w1(const float* w1, const float* b1, const int32_t* fold_table, float* w1m_t, void* stream) {
  if (!w1 || !b1 || !fold_table || !w1m_t) return ARREAU_ERR_NULL;
  fold_w1_t_kernel<<<kMonoPad, kC, 0, (cudaStream_t)stream>>>(w1, b1, fold_table, 258, w1m_t);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_moments(const float* x, const float* sub_cols, int64_t n, double* scratch, double* out,
                              void* stream) {
  if (!x || !scratch || !out) return ARREAU_ERR_NULL;
  if (n <= 0) return ARREAU_ERR_BAD_SHAPE;
  const int blocks = 256;
  moments_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, sub_cols, n, scratch);
  CUDA_LAUNCH_CHECK();
  moments_finish_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(scratch, blocks, out);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

// debug only (not part of the public ABI): per-CTA phase clocks of the persistent TF32 GEMM (GemmArgs::prof)
extern "C" int arreau_debug_set_gemm_prof(long long* prof) {
  g_ws_prof = prof;
  return ARREAU_OK;
}

extern "C" int arreau_sgemm(int32_t a_k_contiguous, int32_t b_k_contiguous, const float* A, int64_t lda, const float* B,
                            int64_t ldb, float* C, int64_t ldc, int32_t M, int32_t N, int64_t K, float alpha,
                            const float* bias, int32_t accumulate, float* partial, int64_t partial_floats, void* stream) {
  if (!A || !B || !C) return ARREAU_ERR_NULL;
  if (M < 0 || N < 0 || K < 0 || (N & 3) || (lda & 3) || (ldb & 3) || (ldc & 3)) return ARREAU_ERR_BAD_SHAPE;
  Gemm g{(cudaStream_t)stream, partial, partial ? (size_t)partial_floats : 0, sm_count()};
  g.tf32 = (a_k_contiguous & 2) || (b_k_contiguous & 2);     // bit 1 of either flag selects the TF32 tensor-core variant
  a_k_contiguous &= 1;
  b_k_contiguous &= 1;
  if (a_k_contiguous && b_k_contiguous) return gemm<true, true>(g, A, lda, B, ldb, C, ldc, M, N, K, alpha, bias, accumulate);
  if (a_k_contiguous) return gemm<true, false>(g, A, lda, B, ldb, C, ldc, M, N, K, alpha, bias, accumulate);
  if (b_k_contiguous) return gemm<false, true>(g, A, lda, B, ldb, C, ldc, M, N, K, alpha, bias, accumulate);
  return gemm<false, false>(g, A, lda, B, ldb, C, ldc, M, N, K, alpha, bias, accumulate);
}

extern "C" int arreau_ponita_backward(const float* params, const arreau_train_layout_t* lay, const arreau_weights* w,
                                      const arreau_workspace* ws, const int32_t* fold_table, const float* x,
                                      const float* vec, const int32_t* row_ptr, const int32_t* src, const int32_t* dst,
                                      const double* dist, const double* dir, const double* lattice,
                                      const int32_t* atom_offset, const int32_t* crystal_of_atom, int32_t N, int32_t G,
                                      double radius, const float* dlogits, const float* dscore, const float* dlen0,
                                      float* workspace, int64_t workspace_bytes, float* grads, int32_t precision,
                                      int32_t forward_kept, void* stream) {
  if (!params || !lay || !w || !ws || !fold_table || !grads || !workspace) return ARREAU_ERR_NULL;
  if (N < 0 || G < 0) return ARREAU_ERR_BAD_SHAPE;
  if (N == 0) return ARREAU_OK;
  if (!ws->h_debug || !ws->x1_debug || !ws->x2_debug || !ws->kernels || !x || !vec || !row_ptr || !src || !dst ||
      !dist || !dir || !lattice || !atom_offset || !crystal_of_atom || !dlogits || !dscore || !dlen0)
    return ARREAU_ERR_NULL;
  const int Z = w->num_states, F = w->num_scalar, V = w->num_vec, R = Z + 4, FV = F + V;
  if (R > 128) return ARREAU_ERR_UNSUPPORTED;
  const int xl_pitch = ((FV + 127) / 128) * 128;
  const long long Ecap = ws->edge_capacity;
  BwdBuffers b = carve(workspace, N, Ecap, xl_pitch);
  if ((int64_t)(b.total * sizeof(float)) > workspace_bytes) return ARREAU_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  if (precision != ARREAU_PRECISION_FP32 && precision != ARREAU_PRECISION_TF32) return ARREAU_ERR_UNSUPPORTED;
  Gemm g{s, b.partial, kPartialFloats, sm_count()};
  g.tf32 = precision == ARREAU_PRECISION_TF32;
  const long long Re = Ecap * kO, Rn = (long long)N * kO;
  const size_t node_elems = (size_t)N * kO * kC, layer_kernel_elems = (size_t)Ecap * kO * kC;
  const int32_t* num_edges_ptr = row_ptr + N;
  const float* P = params;
  float* Gd = grads;
  auto zero = [&](float* p, long long n) -> int {
    if (n <= 0) return ARREAU_OK;
    fill_kernel<<<blocks_for(n, 256), 256, 0, s>>>(p, n, 0.f);
    CUDA_LAUNCH_CHECK();
    return ARREAU_OK;
  };
  auto gelu_f = [&](const float* z, long long rows, int ncols, const float* rs, int rps, float* a) -> int {
    if (rows <= 0) return ARREAU_OK;
    gelu_fwd_kernel<<<blocks_for(rows * ncols / 4, 256), 256, 0, s>>>(z, rows * ncols, ncols, rs, rps, a);
    CUDA_LAUNCH_CHECK();
    return ARREAU_OK;
  };
  auto gelu_b = [&](const float* z, const float* da, long long rows, int ncols, const float* rs, int rps, float* dz) -> int {
    if (rows <= 0) return ARREAU_OK;
    gelu_bwd_kernel<<<blocks_for(rows * ncols / 4, 256), 256, 0, s>>>(z, da, rows * ncols, ncols, rs, rps, dz);
    CUDA_LAUNCH_CHECK();
    return ARREAU_OK;
  };

  // ---- 0. gradient rows of the read-outs, zero dh ---------------------------------------------------------
  TRY(zero(Gd, lay->total));
  TRY(zero(b.dh, (long long)node_elems));
  readout_grad_rows_kernel<<<(unsigned)Rn, 128, 0, s>>>(dlogits, dscore, dlen0, crystal_of_atom, w->ori, N, Z,
                                                        1.0f / (float)(kL * kO), b.dr);
  CUDA_LAUNCH_CHECK();

  // ---- 1. the edge chain (monomials -> z1 -> a1 -> z2 -> kernel basis kb) and the fiber chain ------------
  // (kept in the workspace by arreau_ponita_forward_train; recomputed here after the plain fp32 forward)
  const int Rf = kO * kO;
  if (!forward_kept) {
    TRY(edge_chain_forward(g, b, P, lay, w, fold_table, src, dist, dir, lattice, crystal_of_atom, num_edges_ptr, Ecap, radius));
    TRY(fiber_chain_forward(g, b, P, lay, w->ori, nullptr));
  }
  TRY(zero(b.dfkb, (long long)Rf * kD));

  // ---- 2. layers, last to first -------------------------------------------------------------------------
  for (int l = kL - 1; l >= 0; --l) {
    const float* h_in = ws->h_debug + (size_t)l * node_elems;
    const float* x1 = ws->x1_debug + (size_t)l * node_elems;
    const float* x2 = ws->x2_debug + (size_t)l * node_elems;
    const float* kern = (const float*)ws->kernels + (size_t)l * layer_kernel_elems;
    const float* Wr = P + lay->readout_w + (size_t)l * R * kC;
    const float* W1 = P + lay->lin1_w + (size_t)l * kW * kC;
    const float* W2 = P + lay->lin2_w + (size_t)l * kC * kW;
    const float* Wf = P + lay->conv_fiber_w + (size_t)l * kC * kD;
    const float* ls = P + lay->layer_scale + l * kC;
    // read-out l: r = h_out Wr^T + br   (ponita.py:105); dWr of all layers after the loop
    //   dh += dr Wr      (K = R rows of Wr; dr columns beyond R are zero, so K = R rounded down to the stored rows)
    TRY((gemm<true, false>(g, b.dr, 128, Wr, kC, b.dh, kC, (int)Rn, kC, R, 1.f, nullptr, true)));
    // ConvNext MLP (convnext.py:25-32): y = LN(x2), z = y W1^T + b1, a = gelu(z), m = a W2^T + b2 -- kept per layer by
    // arreau_ponita_forward_train, else recomputed
    const float *yl, *zl, *al, *ml;
    if (forward_kept) {
      yl = b.ys + (size_t)l * Rn * kC; zl = b.zs + (size_t)l * Rn * kW; al = b.as + (size_t)l * Rn * kW;
      ml = b.ms + (size_t)l * Rn * kC;
    } else {
      ln_fwd_kernel<<<blocks_for(Rn * 32, 256), 256, 0, s>>>(x2, P + lay->norm_w + l * kC, P + lay->norm_b + l * kC, Rn, b.y);
      CUDA_LAUNCH_CHECK();
      GemmOpt oz;
      oz.gelu_out = b.a;
      TRY((gemm<true, true>(g, b.y, kC, W1, kC, b.z, kW, (int)Rn, kW, kC, 1.f, P + lay->lin1_b + l * kW, false, oz)));
      TRY((gemm<true, true>(g, b.a, kW, W2, kW, b.m, kC, (int)Rn, kC, kW, 1.f, P + lay->lin2_b + l * kC, false)));
      yl = b.y; zl = b.z; al = b.a; ml = b.m;
    }
    // h_out = h_in + ls * m
    {   // dm = dh * ls, d layer_scale = column sums of dh * m, d lin2 bias = column sums of dm: one pass
      long long sp = (Rn + 63) / 64;
      if (sp > kColSplits) sp = kColSplits;
      ls_bwd_kernel<<<(unsigned)sp, 256, 0, s>>>(b.dh, ml, ls, Rn, b.dm, b.partial);
      CUDA_LAUNCH_CHECK();
      // rows of the second stage's output: [d layer_scale | d lin2 bias] of this layer, lin2_b - layer_scale floats apart
      reduce_partials(s, b.partial, (int)sp, 2 * kC, lay->lin2_b - lay->layer_scale, kC, 1.0f, 0, Gd + lay->layer_scale + l * kC);
      CUDA_LAUNCH_CHECK();
    }
    TRY((gemm<false, false>(g, b.dm, kC, al, kW, Gd + lay->lin2_w + (size_t)l * kC * kW, kW, kC, kW, Rn, 1.f, nullptr, false)));
    {   // dz = (dm W2) * gelu'(z) in the product's epilogue
      GemmOpt od;
      od.gz = zl;
      od.gz_ld = kW;
      od.colsum_out = Gd + lay->lin1_b + l * kW;          // db1 = column sums of dz, from the same epilogue
      TRY((gemm<true, false>(g, b.dm, kC, W2, kW, b.da, kW, (int)Rn, kW, kC, 1.f, nullptr, false, od)));
    }
    TRY((gemm<false, false>(g, b.da, kW, yl, kC, Gd + lay->lin1_w + (size_t)l * kW * kC, kC, kW, kC, Rn, 1.f, nullptr, false)));
    TRY((gemm<true, false>(g, b.da, kW, W1, kC, b.dy, kC, (int)Rn, kC, kW, 1.f, nullptr, false)));
    // LayerNorm backward + conv bias gradient
    {
      int blocks = (int)((Rn + kLnWarps - 1) / kLnWarps);
      if (blocks > kLnBlocks) blocks = kLnBlocks;
      ln_bwd_kernel<<<blocks, kLnWarps * 32, 0, s>>>(x2, b.dy, P + lay->norm_w + l * kC, Rn, b.dx2, b.partial);
      CUDA_LAUNCH_CHECK();
      reduce_partials(s, b.partial, blocks, 3 * kC, 3 * kC, 3 * kC, 1.f, 0, b.small);
      CUDA_LAUNCH_CHECK();
      // b.small[0..383] = [dgamma | dbeta | dbias]
      cudaError_t e = cudaMemcpyAsync(Gd + lay->norm_w + l * kC, b.small, sizeof(float) * kC, cudaMemcpyDeviceToDevice, s);
      if (e == cudaSuccess) e = cudaMemcpyAsync(Gd + lay->norm_b + l * kC, b.small + kC, sizeof(float) * kC, cudaMemcpyDeviceToDevice, s);
      if (e == cudaSuccess) e = cudaMemcpyAsync(Gd + lay->conv_bias + l * kC, b.small + 2 * kC, sizeof(float) * kC, cudaMemcpyDeviceToDevice, s);
      if (e != cudaSuccess) return (int)e;
    }
    // fiber conv backward
    const float* fk = w->fiber_kernel + (size_t)l * kO * kO * kC;
    {
      fiber_bwd_dx1_kernel<<<(N + kDx1Atoms - 1) / kDx1Atoms, kC, 0, s>>>(b.dx2, fk, N, b.dx1);
      CUDA_LAUNCH_CHECK();
      int fb = N < kDfkBlocks ? N : kDfkBlocks;
      fiber_bwd_dfk_kernel<<<fb, 1024, 0, s>>>(x1, b.dx2, N, b.partial);
      CUDA_LAUNCH_CHECK();
      float* dfk = b.dfk + (size_t)l * Rf * kC;
      reduce_partials(s, b.partial, fb, (long long)Rf * kC, Rf * kC, Rf * kC, 1.0f / kO, 0, dfk);
      CUDA_LAUNCH_CHECK();
    }
    // message pass backward: this layer's slab of the kernel gradient, and dh
    if (Re > 0) {
      message_bwd_kernel<<<N + kDkernTailBlocks, 256, 0, s>>>(kern, b.dx1, h_in, row_ptr, src, dst, atom_offset, crystal_of_atom,
                                                            num_edges_ptr, Ecap, N, b.dh, b.dkern + (size_t)l * Re * kC);
      CUDA_LAUNCH_CHECK();
    }
  }
  // read-out weights: dWr_l[R,C] = dr^T h_l for the five layers as ONE product over the kept feature slabs (block-strided
  // operand [Rn][L*C]); dr is 128 wide, only the first R rows of each 128-column block are parameters
  {
    GemmOpt orw;
    orw.b_cblk = (long long)node_elems;
    TRY((gemm<false, false>(g, b.dr, 128, ws->h_debug + node_elems, kC, b.small, kL * kC, 128, kL * kC, Rn, 1.f, nullptr, false, orw)));
    for (int l = 0; l < kL; ++l) {
      cudaError_t e = cudaMemcpy2DAsync(Gd + lay->readout_w + (size_t)l * R * kC, sizeof(float) * kC, b.small + l * kC,
                                        sizeof(float) * kL * kC, sizeof(float) * kC, R, cudaMemcpyDeviceToDevice, s);
      if (e != cudaSuccess) return (int)e;
    }
  }
  // read-out bias: the same dr for every layer -> one column sum, copied to the five slots
  TRY(colsum(g, b.dr, nullptr, Rn, 128, 128, b.small, false));
  for (int l = 0; l < kL; ++l) {
    cudaError_t e = cudaMemcpyAsync(Gd + lay->readout_b + (size_t)l * R, b.small, sizeof(float) * R, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return (int)e;
  }
  // the five layers' kernel projections at once (conv.py:110,113: kernel_l = kb Wk_l^T, fiber_kernel_l = fkb Wf_l^T):
  // the gradient slabs [L][rows][C] are ONE operand [rows][L*C] (block stride = one slab), the weights [L][C][D] one
  // [L*C][D] matrix, so kb / the slabs are streamed once instead of five times and dkb needs no accumulation passes
  {
    GemmOpt of;
    of.a_cblk = (long long)Rf * kC;
    //   dWf[L*C, D] = dfk^T fkb ; dfkb = dfk Wf
    TRY((gemm<false, false>(g, b.dfk, kC, b.fkb, kD, Gd + lay->conv_fiber_w, kD, kL * kC, kD, Rf, 1.f, nullptr, false, of)));
    TRY((gemm<true, false>(g, b.dfk, kC, P + lay->conv_fiber_w, kD, b.dfkb, kD, Rf, kD, kL * kC, 1.f, nullptr, false, of)));
  }

  // ---- 3. node embedding: h0 = x_lift We^T  (ponita.py:98) ------------------------------------------------
  lift_rows_kernel<<<(unsigned)Rn, 256, 0, s>>>(x, vec, w->ori, N, F, V, xl_pitch, b.xl);
  CUDA_LAUNCH_CHECK();
  //   dWe[C, FV] = dh0^T x_lift  (computed xl_pitch wide into scratch, then the FV parameter columns are copied)
  if (xl_pitch > 512) return ARREAU_ERR_UNSUPPORTED;
  TRY((gemm<false, false>(g, b.dh, kC, b.xl, xl_pitch, b.small, xl_pitch, kC, xl_pitch, Rn, 1.f, nullptr, false)));
  {
    cudaError_t e = cudaMemcpy2DAsync(Gd + lay->embed_w, sizeof(float) * FV, b.small, sizeof(float) * xl_pitch, sizeof(float) * FV,
                                      kC, cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return (int)e;
  }

  // ---- 4. edge chain backward ------------------------------------------------------------------------------
  if (Re > 0) {
    GemmOpt ok;
    ok.a_cblk = Re * kC;
    //   dWk[L*C, D] = dkern^T kb
    TRY((gemm<false, false>(g, b.dkern, kC, b.kb, kD, Gd + lay->conv_kernel_w, kD, kL * kC, kD, Re, 1.f, nullptr, false, ok)));
    //   dz2 = (dkern Wk) * gelu'(z2) * window        (b.dkb = dz2)
    ok.gz = b.z2;
    ok.gz_ld = kD;
    ok.rowscale = b.win;
    ok.colsum_out = Gd + lay->basis_b2;                   // db2 = column sums of dz2, from the same epilogue
    TRY((gemm<true, false>(g, b.dkern, kC, P + lay->conv_kernel_w, kD, b.dkb, kD, (int)Re, kD, kL * kC, 1.f, nullptr, false, ok)));
    TRY((gemm<false, false>(g, b.dkb, kD, b.a1, kC, Gd + lay->basis_w2, kC, kD, kC, Re, 1.f, nullptr, false)));
    //   dz1 = (dz2 W2) * gelu'(z1)                   (b.da1 = dz1)
    GemmOpt o1;
    o1.gz = b.z1;
    o1.gz_ld = kC;
    TRY((gemm<true, false>(g, b.dkb, kD, P + lay->basis_w2, kC, b.da1, kC, (int)Re, kC, kD, 1.f, nullptr, false, o1)));
    TRY((gemm<false, false>(g, b.da1, kC, b.mono, 128, b.dw1m, 128, kC, kMonoPad, Re, 1.f, nullptr, false)));
    unfold_w1_grad_kernel<<<kC, 128, 0, s>>>(b.dw1m, fold_table, 258, Gd + lay->basis_w1, Gd + lay->basis_b1);
    CUDA_LAUNCH_CHECK();
  }

  // ---- 5. fiber chain backward -----------------------------------------------------------------------------
  TRY(gelu_b(b.fz2, b.dfkb, Rf, kD, nullptr, 1, b.dfkb));
  TRY(colsum(g, b.dfkb, nullptr, Rf, kD, kD, Gd + lay->fiber_b2, false));
  TRY((gemm<false, false>(g, b.dfkb, kD, b.fa1, kC, Gd + lay->fiber_w2, kC, kD, kC, Rf, 1.f, nullptr, false)));
  {
    GemmOpt o1;
    o1.gz = b.fz1;
    o1.gz_ld = kC;
    TRY((gemm<true, false>(g, b.dfkb, kD, P + lay->fiber_w2, kC, b.fda1, kC, Rf, kC, kD, 1.f, nullptr, false, o1)));
  }
  TRY((gemm<false, false>(g, b.fda1, kC, b.frow, 16, b.fdw16, 16, kC, 16, Rf, 1.f, nullptr, false)));
  unpack_fiber_w1_grad_kernel<<<1, kC, 0, s>>>(b.fdw16, Gd + lay->fiber_w1, Gd + lay->fiber_b1);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

// Training forward with every dense contraction on the generic GEMM (tcgen05 kind::tf32 under ARREAU_PRECISION_TF32) and
// its activations KEPT for arreau_ponita_backward(forward_kept = 1): the edge chain (mono, z1, a1, z2, kb) and the
// LayerNorm output, hidden pre-activation, hidden activation and MLP output of every ConvNext block stay in `workspace`,
// h / x1 / x2 of every layer (h written straight into its kept slab) and the per-layer spatial kernels in `ws` as after
// arreau_ponita_forward with the debug buffers set.  Same mathematics as
// arreau_ponita_forward (ponita/models/ponita.py:88-123); the message pass, fiber conv + LayerNorm, embedding and
// read-outs are the fp32 kernels of that function.
extern "C" int arreau_ponita_forward_train(const float* params, const arreau_train_layout_t* lay, const arreau_weights* w,
                                           const arreau_workspace* ws, const int32_t* fold_table, const float* x,
                                           const float* vec, const int32_t* row_ptr, const int32_t* src, const double* dist,
                                           const double* dir, const double* lattice, const int32_t* atom_offset,
                                           const int32_t* crystal_of_atom, int32_t N, int32_t G, double radius,
                                           float* workspace, int64_t workspace_bytes, int32_t precision, float* logits,
                                           float* score, float* len0, void* stream) {
  if (!params || !lay || !w || !ws || !fold_table || !workspace) return ARREAU_ERR_NULL;
  if (N < 0 || G < 0) return ARREAU_ERR_BAD_SHAPE;
  if (N == 0) return ARREAU_OK;
  if (!ws->h || !ws->y || !ws->acc || !ws->h_debug || !ws->x1_debug || !ws->x2_debug || !ws->kernels || !x || !vec ||
      !row_ptr || !src || !dist || !dir || !lattice || !atom_offset || !crystal_of_atom || !logits || !score || !len0)
    return ARREAU_ERR_NULL;
  if (precision != ARREAU_PRECISION_FP32 && precision != ARREAU_PRECISION_TF32) return ARREAU_ERR_UNSUPPORTED;
  const int Z = w->num_states, F = w->num_scalar, V = w->num_vec, FV = F + V;
  const int xl_pitch = ((FV + 127) / 128) * 128;
  const long long Ecap = ws->edge_capacity;
  BwdBuffers b = carve(workspace, N, Ecap, xl_pitch);
  if ((int64_t)(b.total * sizeof(float)) > workspace_bytes) return ARREAU_ERR_WORKSPACE;
  cudaStream_t s = (cudaStream_t)stream;
  Gemm g{s, b.partial, kPartialFloats, sm_count()};
  g.tf32 = precision == ARREAU_PRECISION_TF32;
  const long long Re = Ecap * kO, Rn = (long long)N * kO;
  const size_t node_elems = (size_t)N * kO * kC, layer_kernel_elems = (size_t)Ecap * kO * kC;
  const float* P = params;
  // embedding (ponita.py:98); the features of layer l live in slab l of h_debug (what the backward reads): no copies
  float* const hs = ws->h_debug;
  if (ws->onehot_types)
    TRY(arreau_node_embed_typed(x, ws->onehot_types, Z, vec, w->w_embed_t, w->ori, N, F, V, hs, stream));
  else
    TRY(arreau_node_embed(x, vec, w->w_embed_t, w->ori, N, F, V, hs, stream));
  // edge chain and the five kernel projections kernels[l] = kb Wk_l^T (conv.py:110) as ONE product: the weights [L][C][D]
  // are one [L*C][D] matrix and the output columns are the per-layer [Re][C] slabs, so kb is streamed once
  TRY(edge_chain_forward(g, b, P, lay, w, fold_table, src, dist, dir, lattice, crystal_of_atom, row_ptr + N, Ecap, radius));
  if (Re > 0) {
    GemmOpt ok;
    ok.c_cblk = (long long)layer_kernel_elems;
    TRY((gemm<true, true>(g, b.kb, kD, P + lay->conv_kernel_w, kD, (float*)ws->kernels, kC, (int)Re, kL * kC, kD, 1.f, nullptr,
                          false, ok)));
  }
  // fiber chain, kept for the backward (the fiber kernels themselves come packed in `w`)
  TRY(fiber_chain_forward(g, b, P, lay, w->ori, nullptr));
  for (int l = 0; l < kL; ++l) {
    const float* kern = (const float*)ws->kernels + (size_t)l * layer_kernel_elems;
    float* yl = b.ys + (size_t)l * Rn * kC;
    float* zl = b.zs + (size_t)l * Rn * kW;
    float* al = b.as + (size_t)l * Rn * kW;
    float* ml = b.ms + (size_t)l * Rn * kC;
    // message pass + fiber conv + bias + LayerNorm (conv.py:111-133, convnext.py:25): y = LN(x2), kept
    const float* h_in = hs + (size_t)l * node_elems;
    float* h_out = hs + (size_t)(l + 1) * node_elems;
    TRY(arreau_message_fiber_norm(kern, 0, h_in, row_ptr, src, w->fiber_kernel + (size_t)l * kO * kO * kC, nullptr,
                                  w->conv_bias + l * kC, w->ln_w + l * kC, w->ln_b + l * kC, N, yl, 0,
                                  ws->x1_debug + l * node_elems, ws->x2_debug + l * node_elems, stream));
    // ConvNext MLP (convnext.py:26-32): z = y W1^T + b1, a = gelu(z) (same epilogue), m = a W2^T + b2, all kept;
    // h_out = h_in + ls * m in the second product's epilogue
    GemmOpt oz;
    oz.gelu_out = al;
    TRY((gemm<true, true>(g, yl, kC, P + lay->lin1_w + (size_t)l * kW * kC, kC, zl, kW, (int)Rn, kW, kC, 1.f,
                          P + lay->lin1_b + l * kW, false, oz)));
    GemmOpt om;
    om.gelu_out = h_out;
    om.res_in = h_in;
    om.res_scale = P + lay->layer_scale + l * kC;
    TRY((gemm<true, true>(g, al, kW, P + lay->lin2_w + (size_t)l * kC * kW, kW, ml, kC, (int)Rn, kC, kW, 1.f,
                          P + lay->lin2_b + l * kC, false, om)));
    TRY(arreau_readout_accumulate(h_out, w->wr_t + (size_t)l * kC * (Z + 4), w->br + l * (Z + 4), w->ori, N, Z, l == 0,
                                  ws->acc, stream));
  }
  TRY(arreau_readout_finalize(ws->acc, atom_offset, N, G, Z, kL, logits, score, len0, stream));
  return ARREAU_OK;
}
