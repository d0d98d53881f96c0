// tcgen05 (fp16 operands, fp32 accumulation in TMEM) kernels for the two GEMM-shaped stages of the step.
//
//   convnext_mlp_tc_kernel   K6     h += layer_scale * (W2 gelu(W1 y + b1) + b2)          convnext.py:26-32
//   edge_kernels_tc_kernel   K3+K4a invariants -> monomials -> basis MLP -> window -> 5 kernel projections
//
// Both are persistent (one CTA per SM, 128-row tiles) and warp specialised:
//   warp 0   producer: cp.async.bulk (TMA engine) of pre-swizzled weight / activation tiles into an mbarrier ring
//   warp 1   MMA issuer: the warp runs the issue loop uniformly, one elected lane issues tcgen05.mma (M = 128, N = 128,
//            K = 16) and tcgen05.commit; the hidden slice (MLP) and the kernel basis (edge) are TENSOR-MEMORY operands
//   warp 2   TMEM allocation / release (MLP: also half of the read-out pooling); warp 3: geometry (edge) / pooling (MLP)
//   warps 4.. epilogue: tcgen05.ld -> bias / GELU / window in registers -> fp16 operand of the next GEMM written back to
//            shared memory in the UMMA layout or to tensor memory (tcgen05.st) -- the intermediates never leave the SM --
//            or the final result to HBM through the TMA engine (bulk stores / bulk reduce-add).  MLP: 16 warps (640
//            threads); edge: a G-group of 16 warps and an L-group of 8 warps working on different jobs (896 threads).
#include "common.cuh"
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int kThreads = 640;
constexpr int kEpiWarp0 = 4;
constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kTileM = 128;
constexpr uint32_t kIdesc128 = umma_idesc_f16(128, 128);

__device__ long long* g_tc_prof = nullptr;   // debug: per-phase clock64 stamps of CTA 0 (scratch/prof_tc.py)
#ifdef ARREAU_TC_PROFILE
#define TC_STAMP(slot)                                                                     \
  do {                                                                                      \
    if (prof && it < 6) prof[(it * 2 + prof_role) * 16 + (slot)] = clock64();               \
  } while (0)
#else
#define TC_STAMP(slot) do { (void)prof; } while (0)
#endif

// 32 accumulator columns -> + bias -> GELU -> four packed fp16 chunks (registers only)
__device__ __forceinline__ void gelu_pack32(const float (&v)[32], const float* __restrict__ bias_s, uint4 (&pk)[4]) {
#pragma unroll
  for (int cc = 0; cc < 4; ++cc) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias_s + cc * 8);
    const float4 b1 = *reinterpret_cast<const float4*>(bias_s + cc * 8 + 4);
    pk[cc].x = gelu2_f16(v[cc * 8 + 0] + b0.x, v[cc * 8 + 1] + b0.y);
    pk[cc].y = gelu2_f16(v[cc * 8 + 2] + b0.z, v[cc * 8 + 3] + b0.w);
    pk[cc].z = gelu2_f16(v[cc * 8 + 4] + b1.x, v[cc * 8 + 5] + b1.y);
    pk[cc].w = gelu2_f16(v[cc * 8 + 6] + b1.z, v[cc * 8 + 7] + b1.w);
  }
}

// =================================================================================================
// K6  ConvNext channel MLP
// =================================================================================================
namespace mlp {
constexpr int kTileBytes = 32768;     // [128 rows x 128 K] fp16 = 2 slabs
constexpr int kWStages = 3;
constexpr int kTilesBytes = (2 + 2 + kWStages) * kTileBytes;
constexpr int kSmemBytes = 232448;    // everything (tiles, bias, barriers) is carved from the dynamic window
constexpr int kChunksPerTile = 8;     // W1_0, W1_1, W2_0, W1_2, W2_1, W1_3, W2_2, W2_3
constexpr uint32_t kHCol = 384;       // TMEM: D1[2] = [0,256), D2 = [256,384), hidden-slice operand H[2] = [384,512) (64 columns each)

struct Bars {
  uint64_t a_full[2], a_empty[2], w_full[kWStages], w_empty[kWStages];
  uint64_t d1_full[2], d1_empty[2], h_full[2], h_empty[2], d2_full, d2_empty;
};
}  // namespace mlp

__global__ void __launch_bounds__(kThreads, 1)
convnext_mlp_tc_kernel(const uint8_t* __restrict__ y_img, const uint8_t* __restrict__ w_img, const float* __restrict__ b1,
                       const float* __restrict__ b2, const float* __restrict__ layer_scale, long long rows,
                       float* __restrict__ h, const float* __restrict__ ori, float* __restrict__ pool_out,
                       const float* __restrict__ pool_wz, int pool_cols) {
  using namespace mlp;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* const A0 = smem;                       // A[ab] = A0 + ab * kTileBytes
  uint8_t* const H0 = smem + 2 * kTileBytes;      // H[b]  = H0 + b * kTileBytes
  uint8_t* const W = smem + 4 * kTileBytes;
  float* const s_b1 = reinterpret_cast<float*>(smem + kTilesBytes);                 // [kW]
  Bars& bars = *reinterpret_cast<Bars*>(smem + kTilesBytes + kW * sizeof(float));
  uint32_t& tmem_base_s = *reinterpret_cast<uint32_t*>(smem + kTilesBytes + kW * sizeof(float) + sizeof(Bars));
  float* const s_ori = reinterpret_cast<float*>(smem + kTilesBytes + kW * sizeof(float) + sizeof(Bars) + 16);   // [kO][3]
  if ((base - smem_u32(smem_raw)) + kTilesBytes + kW * sizeof(float) + sizeof(Bars) + 16 + kO * 3 * sizeof(float) >
      (uint32_t)kSmemBytes)
    __trap();
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform
  const long long tiles = (rows + kTileM - 1) / kTileM;

  for (int i = threadIdx.x; i < kW; i += kThreads) s_b1[i] = b1[i];
  if (pool_out && threadIdx.x < kO * 3) s_ori[threadIdx.x] = ori[threadIdx.x];
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars.a_full[i], 1); mbar_init(&bars.a_empty[i], 1);
      mbar_init(&bars.d1_full[i], 1); mbar_init(&bars.d1_empty[i], kEpiWarps);
      mbar_init(&bars.h_full[i], kEpiWarps); mbar_init(&bars.h_empty[i], 1);
    }
    for (int i = 0; i < kWStages; ++i) { mbar_init(&bars.w_full[i], 1); mbar_init(&bars.w_empty[i], 1); }
    mbar_init(&bars.d2_full, 1); mbar_init(&bars.d2_empty, kEpiWarps);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp == 0 && lane == 0) {
    // ---------------- producer: y tiles and 32 KB weight chunks in the order the MMA warp consumes them.  The first
    // two GEMM1 slices of a tile are issued under the previous tile's tail (see the MMA warp), so per tile the chunk
    // order is W2_0 W1_2 W2_1 W1_3 W2_2 [W1_0 of the next tile] W2_3 [W1_1 of the next tile] ----------------
    uint32_t chunk = 0;
    auto push = [&](int c) {                       // c = chunk index in w_img (W1_0 W1_1 W2_0 W1_2 W2_1 W1_3 W2_2 W2_3)
      const int ws = chunk % kWStages;
      mbar_wait(&bars.w_empty[ws], ((chunk / kWStages) & 1) ^ 1);
      mbar_expect_tx(&bars.w_full[ws], kTileBytes);
      bulk_g2s(W + ws * kTileBytes, w_img + (size_t)c * kTileBytes, kTileBytes, &bars.w_full[ws]);
      ++chunk;
    };
    auto load_y = [&](long long tile, int ti) {
      const int ab = ti & 1;
      mbar_wait(&bars.a_empty[ab], ((ti >> 1) & 1) ^ 1);
      mbar_expect_tx(&bars.a_full[ab], kTileBytes);
      bulk_g2s(A0 + ab * kTileBytes, y_img + (size_t)tile * kTileBytes, kTileBytes, &bars.a_full[ab]);
    };
    if ((long long)blockIdx.x < tiles) {
      load_y(blockIdx.x, 0);
      push(0); push(1);
    }
    int it = 0;
    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const bool has_next = tile + gridDim.x < tiles;
      push(2); push(3); push(4); push(5); push(6);
      if (has_next) {
        load_y(tile + gridDim.x, it + 1);
        push(0);
      }
      push(7);
      if (has_next) push(1);
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer: the whole warp runs the loop uniformly, one elected lane issues
    // (see tc_common.cuh: a divergent single thread pays ~50 cycles per MMA for operand moves) ----------------
    const uint32_t el = elect_one();
    const uint32_t a_lo0 = umma_desc_lo(smem_u32(A0)), w_lo0 = umma_desc_lo(smem_u32(W));
    const uint32_t wfull = smem_u32(&bars.w_full[0]), wempty = smem_u32(&bars.w_empty[0]);
    constexpr uint32_t kSlabLo = 16384 >> 4, kTileLo = kTileBytes >> 4;
    uint32_t ws = 0, wpar = 0;
    int it = 0;
    long long* prof = (blockIdx.x == 0 && el) ? g_tc_prof : nullptr;
    constexpr int prof_role = 0;
    // one 32 KB weight tile (two K slabs): D (+)= X[:, 0:64] . W[0]^T + X[:, 64:128] . W[1]^T, then release it
    auto mma_tile = [&](uint32_t d, uint32_t x_lo, uint32_t accumulate) {
      const uint32_t w_lo = w_lo0 + ws * kTileLo;
      umma_slab_e<4>(d, x_lo, w_lo, kIdesc128, el, accumulate);
      umma_slab_e<4>(d, x_lo + kSlabLo, w_lo + kSlabLo, kIdesc128, el, 1u);
      umma_commit_e(wempty + 8 * ws, el);
      if (++ws == (uint32_t)kWStages) { ws = 0; wpar ^= 1; }
    };
    auto gemm1 = [&](int ti, int j) {        // tile number ti of this CTA: D1[j&1] = y_tile . W1_j^T
      const int b = j & 1, ab = ti & 1;
      const uint32_t use = (uint32_t)ti * 2 + (j >> 1);
      if (j == 0) mbar_wait(&bars.a_full[ab], (ti >> 1) & 1);
      mbar_wait_addr(wfull + 8 * ws, wpar);
      mbar_wait(&bars.d1_empty[b], (use & 1) ^ 1);
      tc_fence_after();
      mma_tile(tmem + b * 128, a_lo0 + ab * kTileLo, 0u);
      umma_commit_e(smem_u32(&bars.d1_full[b]), el);
      if (j == 3) umma_commit_e(smem_u32(&bars.a_empty[ab]), el);
      TC_STAMP(2 + j);
    };
    auto gemm2 = [&](int ti, int j) {        // D2 (+)= H[j&1] . W2_j^T
      const int b = j & 1;
      const uint32_t use = (uint32_t)ti * 2 + (j >> 1);
      mbar_wait_addr(wfull + 8 * ws, wpar);
      mbar_wait(&bars.h_full[b], use & 1);
      if (j == 0) mbar_wait(&bars.d2_empty, (ti & 1) ^ 1);
      tc_fence_after();
      {
        // the hidden slice is the A operand straight out of tensor memory (64 columns of packed fp16 per buffer)
        const uint32_t w_lo = w_lo0 + ws * kTileLo, a_t = tmem + kHCol + b * 64;
        umma_slab_ts_e<4>(tmem + 256, a_t, w_lo, kIdesc128, el, j > 0 ? 1u : 0u);
        umma_slab_ts_e<4>(tmem + 256, a_t + 32, w_lo + kSlabLo, kIdesc128, el, 1u);
        umma_commit_e(wempty + 8 * ws, el);
        if (++ws == (uint32_t)kWStages) { ws = 0; wpar ^= 1; }
      }
      umma_commit_e(smem_u32(&bars.h_empty[b]), el);
      if (j == 3) umma_commit_e(smem_u32(&bars.d2_full), el);
      TC_STAMP(6 + j);
    };
    // Issue order: the first two GEMM1 slices of tile i+1 go in around the last GEMM2 of tile i, so the epilogue warps
    // find slice 0 of the next tile ready while that last GEMM2 runs instead of waiting for it
    if ((long long)blockIdx.x < tiles) { gemm1(0, 0); gemm1(0, 1); }
    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const bool has_next = tile + gridDim.x < tiles;
      TC_STAMP(0);
      gemm2(it, 0); gemm1(it, 2); gemm2(it, 1); gemm1(it, 3); gemm2(it, 2);
      if (has_next) gemm1(it + 1, 0);
      gemm2(it, 3);
      if (has_next) gemm1(it + 1, 1);
    }
  } else if (warp >= kEpiWarp0) {
    // ---------------- epilogue: warp = (lane quarter q, column group cgi of 32 columns) ----------------
    const int q = warp & 3, cgi = (warp - kEpiWarp0) >> 2;
    const int m = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    int it = 0;
    const bool is_issuer = threadIdx.x == kEpiWarp0 * 32;
    long long* prof = (blockIdx.x == 0 && is_issuer) ? g_tc_prof : nullptr;
    constexpr int prof_role = 1;
    // GELU epilogue of hidden slice j of the CTA's tile number `ti`: D1[j & 1] -> + b1 -> GELU -> packed fp16 -> TMEM operand H[j & 1]
    auto gelu_slice = [&](int ti, int j) {
      const int b = j & 1;
      const uint32_t use = (uint32_t)ti * 2 + (j >> 1);
      mbar_wait(&bars.d1_full[b], use & 1);
      mbar_wait(&bars.h_empty[b], (use & 1) ^ 1);
      tc_fence_after();
      float v[32];
      tmem_ld32(tmem + lane_addr + b * 128 + cgi * 32, v);
      uint4 pk[4];
      gelu_pack32(v, s_b1 + j * 128 + cgi * 32, pk);
      {
        // hidden unit k = cgi*32 .. +31 of this 128-slice -> 16 columns of packed pairs in the TMEM operand H[b]
        const uint32_t* pr = reinterpret_cast<const uint32_t*>(pk);
        uint32_t regs[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) regs[i] = pr[i];
        tmem_st16(tmem + lane_addr + kHCol + b * 64 + cgi * 16, regs);
        tmem_wait_st();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&bars.d1_empty[b]);
        mbar_arrive(&bars.h_full[b]);
      }
    };
    // this warp's 32 output channels: lane i keeps b2 and layer_scale of channel cgi*32 + i (broadcast by shuffles in the
    // final epilogue: with 227 KB of shared memory there is no L1 left, every per-tile reload would be an L2 round trip)
    const float my_b2 = __ldg(b2 + cgi * 32 + lane), my_ls = __ldg(layer_scale + cgi * 32 + lane);
    if (blockIdx.x < tiles) gelu_slice(0, 0);
    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      TC_STAMP(0);
      // slice 0 of this tile was done ahead (below / above): it fills the wait for the previous tile's last GEMM
      for (int j = 1; j < 4; ++j) {
        TC_STAMP(1 + 2 * j);
        gelu_slice(it, j);
        TC_STAMP(2 + 2 * j);
      }
      if (tile + gridDim.x < tiles) gelu_slice(it + 1, 0);
      TC_STAMP(9);
      mbar_wait(&bars.d2_full, it & 1);
      tc_fence_after();
      TC_STAMP(10);
      {
        // h += layer_scale * (D2 + b2): the update tile [128 rows x 128 ch] fp32 is 64 KB contiguous in HBM.  It is
        // staged in the two (now idle) H buffers and added into h by the TMA engine (cp.reduce.async.bulk .add.f32:
        // every element is added exactly once, so the result is deterministic) -- no uncoalesced read-modify-write
        // from the SM.  A thread owns 8 16-byte chunks of its row; it writes them in a lane-rotated order
        // (chunk (s + lane) & 7 at step s), which spreads a warp over all banks (4-way = optimal for 512 B).
        float v[32];
        tmem_ld32(tmem + lane_addr + 256 + cgi * 32, v);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.d2_empty);       // accumulators are in registers: release D2 early
        if (it > 0) {
          // the staging area still holds the previous tile's update: its bulk reduce must have finished reading shared
          // memory, and with pooling the pool warps (barriers 3 / 4, one per half) must be done with it too
          if (is_issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          if (!pool_out) {
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
          } else {
            asm volatile("bar.sync 3, %0;" ::"n"(kEpiThreads + 64) : "memory");
            asm volatile("bar.sync 4, %0;" ::"n"(kEpiThreads + 64) : "memory");
          }
        }
        float4 d[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float o4[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float bb = __shfl_sync(0xffffffffu, my_b2, 4 * i + k), ls = __shfl_sync(0xffffffffu, my_ls, 4 * i + k);
            o4[k] = ls * (v[4 * i + k] + bb);
          }
          d[i] = make_float4(o4[0], o4[1], o4[2], o4[3]);
        }
        // barrel-rotate the 8 chunks by r = lane & 7 so that register slot s holds chunk (s + r) & 7
        const int r = lane & 7;
#pragma unroll
        for (int sh = 4; sh >= 1; sh >>= 1) {
          if (r & sh) {
            float4 t[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) t[i] = d[(i + sh) & 7];
#pragma unroll
            for (int i = 0; i < 8; ++i) d[i] = t[i];
          }
        }
        uint8_t* srow = H0 + m * 512 + cgi * 128;
#pragma unroll
        for (int st = 0; st < 8; ++st) *reinterpret_cast<float4*>(srow + (((st + r) & 7) << 4)) = d[st];
        fence_proxy_async();
        if (pool_out) {                                  // staged tile complete -> pool warps
          __threadfence_block();
          asm volatile("bar.arrive 2, %0;" ::"n"(kEpiThreads + 64) : "memory");
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory");
        if (is_issuer) {
          const long long row0 = tile * kTileM;
          const long long left = rows - row0;
          const int valid = (int)(left < kTileM ? left : kTileM);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int n = valid - half * 64 < 64 ? valid - half * 64 : 64;
            if (n > 0)
              asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;" ::"l"(
                               h + (size_t)(row0 + half * 64) * kC),
                           "r"(smem_u32(H0 + half * kTileBytes)), "r"((uint32_t)n * 512u)
                           : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");   // (possibly empty) group per half
          }
        }
      }
      TC_STAMP(11);
    }
    if (is_issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // every update has been added into h
  } else if ((warp == 2 || warp == 3) && pool_out) {
    // ---------------- pooled read-out (see readout_pooled_kernel): the two otherwise idle warps pool the staged residual
    // update over the 16 orientation rows of each of the tile's 8 atoms.  Two phases, one per staging half (rows 0..63 =
    // atoms 0..3, then atoms 4..7), each released to the epilogue warps separately (barriers 3 and 4) so the next
    // tile's H writes are not held up; per phase warp 2 takes the first atom pair, warp 3 the second, lane = 2 channels.
    // Pool entry (include/arreau_b200.h): the orientation mean goes to [group of 16 atoms][C][16 atoms] (a tile is one
    // half of a group); the three vector-pooled parts only meet the score row of the read-out, so this warp contracts
    // them with its 64 channels of that row and leaves 3 partial sums per atom ([atom][2 d + half]) ----------------
    const float* stage = reinterpret_cast<const float*>(H0);
    constexpr float inv = 1.0f / kO;
    const int half = warp - 2;
    const int c2 = half * 64 + lane * 2;                     // this thread's channel pair
    const float wz0 = pool_wz[(size_t)c2 * pool_cols] * inv, wz1 = pool_wz[(size_t)(c2 + 1) * pool_cols] * inv;
    const long long groups = (rows / kO + 15) / 16;
    float* const partials = pool_out + (size_t)groups * kC * 16;
    for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      asm volatile("bar.sync 2, %0;" ::"n"(kEpiThreads + 64) : "memory");
      const bool more = tile + gridDim.x < tiles;            // the last tile has no successor waiting on barriers 3 / 4
      float2 mean[2][4];                                     // [phase][atom of the phase]: (channel c2, c2 + 1)
      float sv[32];                                          // [(phase * 4 + atom) * 3 + d], padded to 32 for the reduction
#pragma unroll
      for (int i = 24; i < 32; ++i) sv[i] = 0.f;
#pragma unroll
      for (int ph = 0; ph < 2; ++ph) {
        float2 acc[3][4];
#pragma unroll
        for (int a = 0; a < 4; ++a) {
          mean[ph][a] = make_float2(0.f, 0.f);
#pragma unroll
          for (int d = 0; d < 3; ++d) acc[d][a] = make_float2(0.f, 0.f);
        }
#pragma unroll 2
        for (int o = 0; o < kO; ++o) {
          const float ox = s_ori[3 * o], oy = s_ori[3 * o + 1], oz = s_ori[3 * o + 2];
          const float2 dx = make_float2(ox, ox), dy = make_float2(oy, oy), dz = make_float2(oz, oz);
#pragma unroll
          for (int a = 0; a < 4; ++a) {
            const float2 v = *reinterpret_cast<const float2*>(stage + ((ph * 4 + a) * kO + o) * kC + c2);
            mean[ph][a].x += v.x; mean[ph][a].y += v.y;
            acc[0][a] = __ffma2_rn(dx, v, acc[0][a]);
            acc[1][a] = __ffma2_rn(dy, v, acc[1][a]);
            acc[2][a] = __ffma2_rn(dz, v, acc[2][a]);
          }
        }
        // done reading this staging half
        if (more) {
          if (ph == 0) asm volatile("bar.arrive 3, %0;" ::"n"(kEpiThreads + 64) : "memory");
          else asm volatile("bar.arrive 4, %0;" ::"n"(kEpiThreads + 64) : "memory");
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int d = 0; d < 3; ++d) sv[(ph * 4 + a) * 3 + d] = fmaf(wz0, acc[d][a].x, wz1 * acc[d][a].y);
      }
      // sum the 24 partial contractions over the warp's lanes: after the five halving exchanges lane i holds value i
#pragma unroll
      for (int bit = 16, n = 32; bit > 0; bit >>= 1, n >>= 1) {
        const bool up = lane & bit;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (j < n / 2) {
            const float send = up ? sv[j] : sv[j + n / 2], keep = up ? sv[j + n / 2] : sv[j];
            sv[j] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
          }
        }
      }
      if (lane < 24) partials[(size_t)(tile * 8 + lane / 3) * 8 + 2 * (lane % 3) + half] = sv[0];
      // the tile's 8 atoms of one channel are one full 32-byte sector of the group's block
      float* const pg = pool_out + (size_t)(tile >> 1) * kC * 16 + (size_t)(tile & 1) * 8;
      float4* p0 = reinterpret_cast<float4*>(pg + (size_t)c2 * 16);
      float4* p1 = reinterpret_cast<float4*>(pg + (size_t)(c2 + 1) * 16);
      p0[0] = make_float4(mean[0][0].x * inv, mean[0][1].x * inv, mean[0][2].x * inv, mean[0][3].x * inv);
      p0[1] = make_float4(mean[1][0].x * inv, mean[1][1].x * inv, mean[1][2].x * inv, mean[1][3].x * inv);
      p1[0] = make_float4(mean[0][0].y * inv, mean[0][1].y * inv, mean[0][2].y * inv, mean[0][3].y * inv);
      p1[1] = make_float4(mean[1][0].y * inv, mean[1][1].y * inv, mean[1][2].y * inv, mean[1][3].y * inv);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// =================================================================================================
// K3 + K4a  edge pipeline
// =================================================================================================
// Per 128-row tile (8 edges x 16 orientations) the tensor pipe runs
//   G1     ACC = monomials [128 x 96] . W1m^T            -> GELU -> hidden tile A2 (shared memory, UMMA image)
//   G2a/b  ACC = hidden [128 x 128] . W2[half]^T         -> + b2, GELU, * window -> kernel basis KB (tensor memory)
//   L0..4  ACC = KB [128 x 256] . Wk_l^T                 -> fp16 -> kernels[l] in HBM (staging + bulk store)
// The kernel basis is a TENSOR-MEMORY operand: the G2 epilogue writes it with tcgen05.st and the five projections (80
// of a tile's 102 MMAs) read it as A from there (tcgen05.mma ... [a_tmem]).  An SS-mode 128 x 128 x 16 MMA reads 8 KB
// of operands per 64 tensor cycles, the shared-memory port's whole 128 B/clk, so a basis in shared memory would leave
// the port no room for the weight ring's writes and the output staging; out of shared memory, it also leaves the space
// for a 5-stage weight ring.
//   TMEM     ACC0 = [0,128): G jobs, ACC1 = [128,256): L jobs; KB0 = [256,384), KB1 = [384,512): kernel basis of the
//            current / the next tile (packed fp16 pairs)
//   jobs     MMA issue order per tile i: L0 G1' L1 G2a' L2 G2b' L3 L4 (' = tile i+1), so the head of the next tile runs
//            under this tile's projections
//   ring     Wk0 W1' Wk1 W2a' Wk2 W2b' Wk3 Wk4  (13 chunks of 32 KB per tile, 5 stages)
// The jobs are drained by two epilogue groups with one accumulator slot each, working at the same time:
//   G-group (warps 4..19)   gen' -> G1' (GELU -> hidden tile A2) -> G2a', G2b' (GELU * window -> kernel basis in TMEM)
//   L-group (warps 20..27)  L0 .. L4: fp16 pack -> staging -> bulk store of kernels[l]  (64 columns per thread)
// A group pulls a finished accumulator into registers and hands the slot back before its post-processing, so the
// tensor pipe runs ahead of both.  Every producer/consumer chain of the tile head (monomials, hidden layer, kernel
// basis) stays inside the G-group, so no cross-group hand-off is needed: completion of earlier MMAs is implied by the
// in-order tensor pipe (a finished GEMM2 says that the previous tile's five projections have finished reading the
// other kernel-basis buffer).  Warp 3 computes the per-edge geometry up to two tiles ahead.
// 896 threads (a block holds at most 1024) -> at most 73 registers per thread.
// The earlier version with a single epilogue group is at commit be8d4ea; profiles/r2_ab_edge_variants.txt has the A/B
// of the two.
namespace edge {
constexpr int kEdgesPerTile = kTileM / kO;
constexpr int kGeo = 12;                // floats per edge: dir (3), dist, cos(dir, a/b/c) (3), window, valid, pad
constexpr int kChunkBytes = 32768;
constexpr int kStages = 5;
constexpr int kStageBytes = 32768;
constexpr int kA2Bytes = 32768;
constexpr int kTilesBytes = kA2Bytes + kStageBytes + kStages * kChunkBytes;
constexpr int kSmemBytes = 232448;
constexpr uint32_t kKbCol = 256;
constexpr int kLWarps = 8;                 // L-group: 4 lane quarters x 2 column halves
constexpr int kEdgeThreads = (kEpiWarp0 + kEpiWarps + kLWarps) * 32;   // 896: 4 service warps + G-group (16) + L-group (8)
constexpr int kLWarp0 = kEpiWarp0 + kEpiWarps;

struct Bars {
  uint64_t w_full[kStages], w_empty[kStages];
  uint64_t a1_full, a2_full;
  uint64_t acc_full[2], acc_empty[2];      // [0] = G jobs (ACC0), [1] = L jobs (ACC1)
  uint64_t kb_full[2];
  uint64_t g_full[2], g_empty[2];
};

// monomial n of csrc/common.cuh monomials83 as compile-time index triples; 83 = constant 1 (bias), > 83 = 0
struct MonoIdx { int deg, a, b, c; };
__host__ __device__ constexpr MonoIdx mono_idx(int n) {
  if (n < 6) return {1, n, 0, 0};
  int m = 6;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) {
      if (m == n) return {2, i, j, 0};
      ++m;
    }
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j)
      for (int k = j; k < 6; ++k) {
        if (m == n) return {3, i, j, k};
        ++m;
      }
  return {n == kMono ? 0 : -1, 0, 0, 0};
}
template <int N>
__device__ __forceinline__ float mono_val(const float (&v)[6], float one) {
  constexpr MonoIdx mi = mono_idx(N);
  if constexpr (mi.deg == 1) return v[mi.a];
  else if constexpr (mi.deg == 2) return v[mi.a] * v[mi.b];
  else if constexpr (mi.deg == 3) return v[mi.a] * v[mi.b] * v[mi.c];
  else if constexpr (mi.deg == 0) return one;
  else return 0.f;
}
template <int C>
__device__ __forceinline__ uint4 mono_chunk(const float (&v)[6], float one) {
  uint4 pk;
  pk.x = pack_f16(mono_val<C * 8 + 0>(v, one), mono_val<C * 8 + 1>(v, one));
  pk.y = pack_f16(mono_val<C * 8 + 2>(v, one), mono_val<C * 8 + 3>(v, one));
  pk.z = pack_f16(mono_val<C * 8 + 4>(v, one), mono_val<C * 8 + 5>(v, one));
  pk.w = pack_f16(mono_val<C * 8 + 6>(v, one), mono_val<C * 8 + 7>(v, one));
  return pk;
}
// chunks 3*PART .. 3*PART+2 of monomial row m (12 chunks of 8 = 96 columns; slab = chunk / 8)
template <int PART>
__device__ __forceinline__ void store_mono_part(const float (&v)[6], float one, uint8_t* a1, int m) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    constexpr int kBase = PART * 3;
    const int c = kBase + i;
    uint4 pk = i == 0 ? mono_chunk<kBase>(v, one) : (i == 1 ? mono_chunk<kBase + 1>(v, one) : mono_chunk<kBase + 2>(v, one));
    *reinterpret_cast<uint4*>(a1 + (c >> 3) * 16384 + m * kRowBytes + (((c & 7) ^ (m & 7)) << 4)) = pk;
  }
}

}  // namespace edge

__global__ void __launch_bounds__(edge::kEdgeThreads, 1)
edge_kernels_tc_kernel(const double* __restrict__ dir, const double* __restrict__ dist, const double* __restrict__ lattice,
                        const int32_t* __restrict__ crystal_of_atom, const int32_t* __restrict__ src,
                        const int32_t* __restrict__ num_edges_ptr, long long edge_capacity, const float* __restrict__ ori,
                        const uint8_t* __restrict__ w1_img, const uint8_t* __restrict__ w_img, const float* __restrict__ b2,
                        double radius, __half* __restrict__ kernels) {
  using namespace edge;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  float* const s_b2 = reinterpret_cast<float*>(smem + kTilesBytes);                                   // [kD]
  float* const s_geo = s_b2 + kD;                                                                      // [2][8 edges][kGeo]
  Bars& bars = *reinterpret_cast<Bars*>(smem + kTilesBytes + (kD + 2 * kEdgesPerTile * kGeo) * sizeof(float));
  uint32_t& tmem_base_s =
      *reinterpret_cast<uint32_t*>(smem + kTilesBytes + (kD + 2 * kEdgesPerTile * kGeo) * sizeof(float) + sizeof(Bars));
  if ((base - smem_u32(smem_raw)) + kTilesBytes + (kD + 2 * kEdgesPerTile * kGeo) * sizeof(float) + sizeof(Bars) + 16 > (uint32_t)kSmemBytes)
    __trap();
  uint8_t* const A2 = smem;                   // monomial tile A1, then the hidden layer
  uint8_t* const S = A2 + kA2Bytes;           // two 16 KB halves (rows 0..63 / 64..127) of one layer's output tile
  uint8_t* const W = S + kStageBytes;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform
  long long E = *num_edges_ptr;
  if (E > edge_capacity) E = edge_capacity;
  const long long tiles = (E + kEdgesPerTile - 1) / kEdgesPerTile;
  const long long first = blockIdx.x, stride = gridDim.x;

  for (int i = threadIdx.x; i < kD; i += kEdgeThreads) s_b2[i] = b2[i];
  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&bars.w_full[i], 1); mbar_init(&bars.w_empty[i], 1); }
    mbar_init(&bars.a1_full, kEpiWarps); mbar_init(&bars.a2_full, kEpiWarps);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars.acc_full[i], 1); mbar_init(&bars.acc_empty[i], i == 0 ? kEpiWarps : kLWarps);
      mbar_init(&bars.kb_full[i], 2 * kEpiWarps);            // both output halves of GEMM2
      mbar_init(&bars.g_full[i], 1); mbar_init(&bars.g_empty[i], kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp == 3) {
    // ---------------- geometry: the per-edge part of the invariants, up to two tiles ahead ----------------
    uint32_t k = 0;
    for (long long tile = first; tile < tiles; tile += stride, ++k) {
      const int buf = k & 1;
      mbar_wait(&bars.g_empty[buf], ((k >> 1) & 1) ^ 1);
      if (lane < kEdgesPerTile) {
        const long long e = tile * kEdgesPerTile + lane;
        float* gp = s_geo + (buf * kEdgesPerTile + lane) * kGeo;
        float vals[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (e < E) {
          const double* lat9 = lattice + 9 * (size_t)crystal_of_atom[src[e]];
          const float dx = (float)dir[3 * e], dy = (float)dir[3 * e + 1], dz = (float)dir[3 * e + 2];
          const float dd = dx * dx + dy * dy + dz * dz;
          vals[0] = dx; vals[1] = dy; vals[2] = dz;
          vals[3] = (float)dist[e];
#pragma unroll
          for (int mm = 0; mm < 3; ++mm) {
            const float ax = (float)lat9[3 * mm], ay = (float)lat9[3 * mm + 1], az = (float)lat9[3 * mm + 2];
            const float w12 = dx * ax + dy * ay + dz * az, w2 = ax * ax + ay * ay + az * az;
            vals[4 + mm] = w12 * rsqrtf(fmaxf(dd * w2, 1e-16f));     // CosineSimilarity, eps = 1e-8
          }
          vals[7] = cutoff_window(dist[e], radius);
          vals[8] = 1.0f;
        }
#pragma unroll
        for (int i = 0; i < 9; ++i) gp[i] = vals[i];
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.g_full[buf]);
    }
  } else if (warp == 0 && lane == 0) {
    // ---------------- producer: 32 KB weight chunks in the order the MMA warp consumes them ----------------
    if (first < tiles) {
      uint32_t st = 0, par = 1;          // waits on w_empty start at parity 1 (a fresh barrier passes)
      auto push = [&](const uint8_t* src_chunk) {
        mbar_wait(&bars.w_empty[st], par);
        mbar_expect_tx(&bars.w_full[st], kChunkBytes);
        bulk_g2s(W + st * kChunkBytes, src_chunk, kChunkBytes, &bars.w_full[st]);
        if (++st == kStages) { st = 0; par ^= 1; }
      };
      auto push_w = [&](int c0, int n) { for (int c = c0; c < c0 + n; ++c) push(w_img + (size_t)c * kChunkBytes); };
      push(w1_img);
      push_w(0, 2);                                   // first tile: W1, W2 (both output halves)
      for (long long tile = first; tile < tiles; tile += stride) {
        const bool has_next = tile + stride < tiles;
        push_w(2, 2);                                 // Wk_0
        if (has_next) push(w1_img);
        push_w(4, 2);                                 // Wk_1
        if (has_next) push_w(0, 1);                   // W2, output half 0
        push_w(6, 2);                                 // Wk_2
        if (has_next) push_w(1, 1);                   // W2, output half 1
        push_w(8, 4);                                 // Wk_3, Wk_4
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (warp-uniform, one elected lane; see the MLP kernel) ----------------
    if (first < tiles) {
      const uint32_t el = elect_one();
      const uint32_t a2_lo = umma_desc_lo(smem_u32(A2)), w_lo = umma_desc_lo(smem_u32(W));
      const uint32_t wfull = smem_u32(&bars.w_full[0]), wempty = smem_u32(&bars.w_empty[0]);
      const uint32_t accfull = smem_u32(&bars.acc_full[0]), accempty = smem_u32(&bars.acc_empty[0]);
      constexpr uint32_t kSlabLo = 16384 >> 4;
      uint32_t st = 0, par = 0, ug = 0, ul = 0;        // uses of the G slot (ACC0) / the L slot (ACC1) so far
      // debug: clock64 stamps of CTA 0, tiles 2..9 of this CTA: [tile][role 0 = MMA][3 * job + {entry, waits done, issued}]
      long long* const prof = (blockIdx.x == 0 && el) ? g_tc_prof : nullptr;
      uint32_t pit = 0, pjob = 0;
#ifdef ARREAU_TC_PROFILE
      auto stamp = [&](int what) { if (prof && pit >= 2 && pit < 10) prof[((pit - 2) * 3 + 0) * 32 + 3 * pjob + what] = clock64(); };
#else
      auto stamp = [&](int) { (void)prof; };
#endif
      auto advance = [&]() { if (++st == kStages) { st = 0; par ^= 1; } };
      // accumulator slot of a job: wait until its group has pulled the slot's previous content into registers
      auto acc_begin = [&](uint32_t slot) -> uint32_t {
        mbar_wait_addr(accempty + 8 * slot, ((slot ? ul : ug) & 1u) ^ 1u);
        tc_fence_after();
        return tmem + slot * 128;
      };
      auto acc_end = [&](uint32_t slot) { umma_commit_e(accfull + 8 * slot, el); if (slot) ++ul; else ++ug; };
      // one ring chunk = two K slabs, A from shared memory (GEMM1 / GEMM2)
      auto pair_ss = [&](uint32_t d, uint32_t a_lo, int ksteps1) {
        mbar_wait_addr(wfull + 8 * st, par);
        const uint32_t b_lo = w_lo + st * (2 * kSlabLo);
        umma_slab_e<4>(d, a_lo, b_lo, kIdesc128, el, 0u);
        if (ksteps1 == 4) umma_slab_e<4>(d, a_lo + kSlabLo, b_lo + kSlabLo, kIdesc128, el, 1u);
        else umma_slab_e<2>(d, a_lo + kSlabLo, b_lo + kSlabLo, kIdesc128, el, 1u);
        umma_commit_e(wempty + 8 * st, el);
        advance();
      };
      // one ring chunk = two K slabs (128 K values = 64 TMEM columns of packed pairs), A from tensor memory (GEMM3)
      auto pair_ts = [&](uint32_t d, uint32_t a_t, uint32_t accumulate) {
        mbar_wait_addr(wfull + 8 * st, par);
        const uint32_t b_lo = w_lo + st * (2 * kSlabLo);
        umma_slab_ts_e<4>(d, a_t, b_lo, kIdesc128, el, accumulate);
        umma_slab_ts_e<4>(d, a_t + 32, b_lo + kSlabLo, kIdesc128, el, 1u);
        umma_commit_e(wempty + 8 * st, el);
        advance();
      };
      auto gemm1 = [&](uint32_t k) {       // ACC = A1[128 x 96] . W1m^T   (tile ordinal k)
        stamp(0);
        mbar_wait(&bars.a1_full, k & 1);
        const uint32_t d = acc_begin(0);
        stamp(1);
        pair_ss(d, a2_lo, 2);
        acc_end(0);
        stamp(2); ++pjob;
      };
      auto gemm2 = [&](uint32_t k, int nh) {   // ACC = hidden[128 x 128] . W2[nh]^T
        stamp(0);
        if (nh == 0) mbar_wait(&bars.a2_full, k & 1);
        const uint32_t d = acc_begin(0);
        stamp(1);
        pair_ss(d, a2_lo, 4);
        acc_end(0);
        stamp(2); ++pjob;
      };
      gemm1(0);
      gemm2(0, 0);
      gemm2(0, 1);
      uint32_t it = 0;
      for (long long tile = first; tile < tiles; tile += stride, ++it) {
        const bool has_next = tile + stride < tiles;
        const uint32_t kb = tmem + kKbCol + (it & 1u) * 128;
        pit = it; pjob = 0;
#pragma unroll 1
        for (int l = 0; l < kL; ++l) {
          stamp(0);
          const uint32_t d = acc_begin(1);
          if (l == 0) {                        // kernel basis of this tile is in tensor memory
            mbar_wait(&bars.kb_full[it & 1u], (it >> 1) & 1u);
            tc_fence_after();
          }
          stamp(1);
          pair_ts(d, kb, 0u);
          pair_ts(d, kb + 64, 1u);
          acc_end(1);
          stamp(2); ++pjob;
          if (has_next) {
            if (l == 0) gemm1(it + 1);
            else if (l == 1) gemm2(it + 1, 0);
            else if (l == 2) gemm2(it + 1, 1);
          }
        }
      }
    }
  } else if (warp >= kEpiWarp0 && warp < kLWarp0) {
    // ---------------- G-group: generator + the two GELU epilogues; warp = (lane quarter q, column group cgi) --------
    const int q = warp & 3, cgi = (warp - kEpiWarp0) >> 2;
    const int m = q * 32 + lane;                     // tile row = (edge m / 16, orientation m % 16)
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const float ox = ori[3 * (m & 15)], oy = ori[3 * (m & 15) + 1], oz = ori[3 * (m & 15) + 2];
    float win_cur = 0.f;
    uint32_t ug = 0;
    long long* const prof = (blockIdx.x == 0 && threadIdx.x == kEpiWarp0 * 32) ? g_tc_prof : nullptr;
    uint32_t pit = 0, pjob = 0;
#ifdef ARREAU_TC_PROFILE
    auto stamp = [&](int what) { if (prof && pit >= 2 && pit < 10) prof[((pit - 2) * 3 + 1) * 32 + 3 * pjob + what] = clock64(); };
#else
    auto stamp = [&](int) { (void)prof; };
#endif
    auto acc_wait = [&]() {
      stamp(0);
      mbar_wait(&bars.acc_full[0], ug & 1u);
      tc_fence_after();
    };
    auto acc_release = [&]() {                       // the accumulator is in registers: hand the slot back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.acc_empty[0]);
      ++ug;
      stamp(1);
    };
    auto ld32 = [&](uint32_t (&r0)[16], uint32_t (&r1)[16]) {      // columns cgi*32 .. +31 of row m, one wait for both
      tmem_ld16_nowait(tmem + lane_addr + cgi * 32, r0);
      tmem_ld16_nowait(tmem + lane_addr + cgi * 32 + 16, r1);
      tmem_wait_ld();
    };
    auto gen = [&](uint32_t k) {                     // monomials of tile ordinal k -> A2 (GEMM1's A operand A1)
      const int buf = k & 1;
      mbar_wait(&bars.g_full[buf], (k >> 1) & 1);
      const float* gp = s_geo + (buf * kEdgesPerTile + (m >> 4)) * kGeo;
      const float dx = gp[0], dy = gp[1], dz = gp[2];
      float attr[6];
      const float i1 = dx * ox + dy * oy + dz * oz;
      const float px = dx - i1 * ox, py = dy - i1 * oy, pz = dz - i1 * oz;
      attr[0] = i1;
      attr[1] = sqrtf(px * px + py * py + pz * pz);
      attr[2] = gp[3]; attr[3] = gp[4]; attr[4] = gp[5]; attr[5] = gp[6];
      win_cur = gp[7];
      const float one = gp[8];
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.g_empty[buf]);
      switch (cgi) {
        case 0: store_mono_part<0>(attr, one, A2, m); break;
        case 1: store_mono_part<1>(attr, one, A2, m); break;
        case 2: store_mono_part<2>(attr, one, A2, m); break;
        default: store_mono_part<3>(attr, one, A2, m); break;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.a1_full);
    };
    auto job_g1 = [&]() {                            // hidden = GELU(GEMM1) -> A2 (unit cgi*32.. -> slab cgi>>1)
      uint32_t v0[16], v1[16];
      acc_wait();
      ld32(v0, v1);
      acc_release();
      uint8_t* row = A2 + (cgi >> 1) * 16384 + m * kRowBytes;
      const int chunk0 = (cgi & 1) * 4;
      auto f = [](uint32_t u) { return __uint_as_float(u); };
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        uint4 pk;
        pk.x = gelu2_f16(f(v0[cc * 8 + 0]), f(v0[cc * 8 + 1])); pk.y = gelu2_f16(f(v0[cc * 8 + 2]), f(v0[cc * 8 + 3]));
        pk.z = gelu2_f16(f(v0[cc * 8 + 4]), f(v0[cc * 8 + 5])); pk.w = gelu2_f16(f(v0[cc * 8 + 6]), f(v0[cc * 8 + 7]));
        *reinterpret_cast<uint4*>(row + (((chunk0 + cc) ^ (m & 7)) << 4)) = pk;
      }
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        uint4 pk;
        pk.x = gelu2_f16(f(v1[cc * 8 + 0]), f(v1[cc * 8 + 1])); pk.y = gelu2_f16(f(v1[cc * 8 + 2]), f(v1[cc * 8 + 3]));
        pk.z = gelu2_f16(f(v1[cc * 8 + 4]), f(v1[cc * 8 + 5])); pk.w = gelu2_f16(f(v1[cc * 8 + 6]), f(v1[cc * 8 + 7]));
        *reinterpret_cast<uint4*>(row + (((chunk0 + 2 + cc) ^ (m & 7)) << 4)) = pk;
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.a2_full);
      stamp(2); ++pjob;
    };
    auto job_g2 = [&](uint32_t k, int nh) {          // kernel basis half nh of tile k -> KB[k & 1] (tensor memory)
      uint32_t v0[16], v1[16];
      acc_wait();
      ld32(v0, v1);
      acc_release();
      const __half2 sc = __float2half2_rn(win_cur);
      const float* bias = s_b2 + nh * 128 + cgi * 32;
      const uint32_t dst = tmem + kKbCol + (k & 1u) * 128 + lane_addr + nh * 64 + cgi * 16;
      // in place: packed pair i of the 32 columns overwrites v0[i] (its inputs v0[2i], v0[2i+1] / v1[..] are dead by then)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 b = *reinterpret_cast<const float2*>(bias + 2 * i);           // warp-uniform: smem broadcast
        v0[i] = gelu2_scaled_f16(__uint_as_float(v0[2 * i]) + b.x, __uint_as_float(v0[2 * i + 1]) + b.y, sc);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float2 b = *reinterpret_cast<const float2*>(bias + 16 + 2 * i);
        v0[8 + i] = gelu2_scaled_f16(__uint_as_float(v1[2 * i]) + b.x, __uint_as_float(v1[2 * i + 1]) + b.y, sc);
      }
      tmem_st16(dst, v0);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars.kb_full[k & 1u]);
      stamp(2); ++pjob;
    };
    if (first < tiles) {
      gen(0);
      job_g1();
      job_g2(0, 0);
      job_g2(0, 1);
      uint32_t it = 0;
      for (long long tile = first; tile < tiles; tile += stride, ++it) {
        if (tile + stride >= tiles) break;
        pit = it; pjob = 0;
#ifdef ARREAU_TC_PROFILE
        if (prof && pit >= 2 && pit < 10) prof[((pit - 2) * 3 + 1) * 32 + 30] = clock64();
#endif
        gen(it + 1);                               // A2 is free: this group has drained both halves of tile it's GEMM2
#ifdef ARREAU_TC_PROFILE
        if (prof && pit >= 2 && pit < 10) prof[((pit - 2) * 3 + 1) * 32 + 31] = clock64();
#endif
        job_g1();
        job_g2(it + 1, 0);
        job_g2(it + 1, 1);
      }
    }
  } else if (warp >= kLWarp0) {
    // ---------------- L-group: kernels[l][e][o][c] = ACC1 (fp16), staged in shared memory, bulk stores ---------------
    // warp = (lane quarter q, column half ch): row m, channels ch*64 .. +63, pulled in two passes of 32 columns
    const int q = warp & 3, ch = (warp - kLWarp0) >> 2;
    const int m = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int hf = q >> 1;                           // staging half of this warp's rows
    const bool is_issuer = ch == 0 && (q & 1) == 0 && lane == 0;      // one bulk-store issuer per half tile
    uint32_t ul = 0;
    long long* const prof = (blockIdx.x == 0 && threadIdx.x == kLWarp0 * 32) ? g_tc_prof : nullptr;
    uint32_t pit = 0, pjob = 0;
#ifdef ARREAU_TC_PROFILE
    auto stamp = [&](int what) { if (prof && pit >= 2 && pit < 10) prof[((pit - 2) * 3 + 2) * 32 + 3 * pjob + what] = clock64(); };
#else
    auto stamp = [&](int) { (void)prof; };
#endif
    auto pack16 = [](const uint32_t (&r)[16], uint4 (&pk)[2]) {
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        pk[cc].x = pack_f16(__uint_as_float(r[cc * 8 + 0]), __uint_as_float(r[cc * 8 + 1]));
        pk[cc].y = pack_f16(__uint_as_float(r[cc * 8 + 2]), __uint_as_float(r[cc * 8 + 3]));
        pk[cc].z = pack_f16(__uint_as_float(r[cc * 8 + 4]), __uint_as_float(r[cc * 8 + 5]));
        pk[cc].w = pack_f16(__uint_as_float(r[cc * 8 + 6]), __uint_as_float(r[cc * 8 + 7]));
      }
    };
    auto job_layer = [&](int l, long long tile) {
      stamp(0);
      mbar_wait(&bars.acc_full[1], ul & 1u);
      tc_fence_after();
      const uint32_t acc = tmem + 128 + lane_addr + ch * 64;
      uint4 pk[8];                                   // 64 channels of row m as packed fp16
      {
        uint32_t r0[16], r1[16];
        tmem_ld16_nowait(acc, r0);
        tmem_ld16_nowait(acc + 16, r1);
        tmem_wait_ld();
        pack16(r0, *reinterpret_cast<uint4(*)[2]>(&pk[0]));
        pack16(r1, *reinterpret_cast<uint4(*)[2]>(&pk[2]));
        tmem_ld16_nowait(acc + 32, r0);
        tmem_ld16_nowait(acc + 48, r1);
        tmem_wait_ld();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.acc_empty[1]);      // the accumulator is in registers: hand the slot back
        ++ul;
        stamp(1);
        pack16(r0, *reinterpret_cast<uint4(*)[2]>(&pk[4]));
        pack16(r1, *reinterpret_cast<uint4(*)[2]>(&pk[6]));
      }
      uint8_t* stage = S + hf * 16384;
      if (is_issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // this half's previous store has left smem
      asm volatile("bar.sync %0, %1;" ::"r"(1 + hf), "n"(kLWarps * 32 / 2) : "memory");
      uint8_t* orow = stage + (m & 63) * 256;
#pragma unroll
      for (int cc = 0; cc < 8; ++cc) *reinterpret_cast<uint4*>(orow + (((ch * 8 + cc) ^ (m & 15)) << 4)) = pk[cc];
      fence_proxy_async();
      asm volatile("bar.sync %0, %1;" ::"r"(1 + hf), "n"(kLWarps * 32 / 2) : "memory");
      if (is_issuer) {
        const long long left = E - tile * kEdgesPerTile - hf * (kEdgesPerTile / 2);   // edges of this half still valid
        if (left > 0) {
          const uint32_t bytes = (uint32_t)(left < kEdgesPerTile / 2 ? left : kEdgesPerTile / 2) * (kO * kC * 2);
          __half* out = kernels + ((size_t)l * edge_capacity * kO + (size_t)tile * kTileM + hf * 64) * kC;
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(out), "r"(smem_u32(stage)), "r"(bytes)
                       : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
      stamp(2); ++pjob;
    };
    if (first < tiles) {
      uint32_t it = 0;
      for (long long tile = first; tile < tiles; tile += stride, ++it) {
        pit = it; pjob = 0;
#pragma unroll 1
        for (int l = 0; l < kL; ++l) job_layer(l, tile);
      }
      if (is_issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // all output tiles have landed
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

int num_sms_tc() {
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

// debug only (not part of the public ABI): clock64 stamps of CTA 0 of the MLP and edge kernels (ARREAU_TC_PROFILE builds)
extern "C" int arreau_debug_set_tc_profile(long long* buf) {
  return (int)cudaMemcpyToSymbol(g_tc_prof, &buf, sizeof(buf));
}

static int convnext_mlp_f16_launch(const void* y_img, const void* w_img, const float* b1, const float* b2,
                                   const float* layer_scale, int64_t num_rows, float* h, const float* ori,
                                   float* pool_out, const float* pool_wz, int pool_cols, void* stream) {
  if (num_rows == 0) return ARREAU_OK;
  if (!y_img || !w_img || !b1 || !b2 || !layer_scale || !h) return ARREAU_ERR_NULL;
  if (num_rows < 0 || (pool_out && num_rows % kO != 0)) return ARREAU_ERR_BAD_SHAPE;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(convnext_mlp_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, mlp::kSmemBytes);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  const long long tiles = (num_rows + kTileM - 1) / kTileM;
  const int grid = (int)(tiles < (long long)num_sms_tc() ? tiles : (long long)num_sms_tc());
  convnext_mlp_tc_kernel<<<grid, kThreads, mlp::kSmemBytes, (cudaStream_t)stream>>>(
      (const uint8_t*)y_img, (const uint8_t*)w_img, b1, b2, layer_scale, (long long)num_rows, h, ori, pool_out, pool_wz,
      pool_cols);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

extern "C" int arreau_convnext_mlp_f16(const void* y_img, const void* w_img, const float* b1, const float* b2,
                                        const float* layer_scale, int64_t num_rows, float* h, void* stream) {
  return convnext_mlp_f16_launch(y_img, w_img, b1, b2, layer_scale, num_rows, h, nullptr, nullptr, nullptr, 0, stream);
}

extern "C" int arreau_convnext_mlp_f16_pooled(const void* y_img, const void* w_img, const float* b1, const float* b2,
                                               const float* layer_scale, int64_t num_rows, float* h, const float* ori,
                                               float* pool_out, const float* readout_v_k, int32_t num_states,
                                               void* stream) {
  if (num_rows > 0 && (!ori || !pool_out || !readout_v_k)) return ARREAU_ERR_NULL;
  if (num_states <= 0) return ARREAU_ERR_BAD_SHAPE;
  // the spare warps contract the vector-pooled parts with column Z of the entry's [C][Z+6] read-out matrix
  return convnext_mlp_f16_launch(y_img, w_img, b1, b2, layer_scale, num_rows, h, ori, pool_out, readout_v_k + num_states,
                                 num_states + 6, stream);
}

extern "C" int arreau_edge_kernels_f16(const double* dir, const double* dist, const double* lattice,
                                        const int32_t* crystal_of_atom, const int32_t* src, const int32_t* num_edges_ptr,
                                        int64_t edge_capacity, const float* ori, const void* w1_img, const void* w_img,
                                        const float* b2, double radius, void* kernels_f16, void* stream) {
  if (edge_capacity == 0) return ARREAU_OK;
  if (!dir || !dist || !lattice || !crystal_of_atom || !src || !num_edges_ptr || !ori || !w1_img || !w_img || !b2 ||
      !kernels_f16)
    return ARREAU_ERR_NULL;
  if (edge_capacity < 0) return ARREAU_ERR_BAD_SHAPE;
  const long long tiles = (edge_capacity + edge::kEdgesPerTile - 1) / edge::kEdgesPerTile;
  const int grid = (int)(tiles < (long long)num_sms_tc() ? tiles : (long long)num_sms_tc());
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(edge_kernels_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, edge::kSmemBytes);
    if (e != cudaSuccess) return (int)e;
    attr_set = true;
  }
  edge_kernels_tc_kernel<<<grid, edge::kEdgeThreads, edge::kSmemBytes, (cudaStream_t)stream>>>(
      dir, dist, lattice, crystal_of_atom, src, num_edges_ptr, (long long)edge_capacity, ori, (const uint8_t*)w1_img,
      (const uint8_t*)w_img, b2, radius, (__half*)kernels_f16);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}
