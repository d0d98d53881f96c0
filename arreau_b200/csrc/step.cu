// Host-side orchestration of the step behind the C ABI: the Ponita forward (K2..K7) and the whole
// denoise step (K9 + K1 + forward + K8) as a fixed sequence of launches on one stream.  No host
// synchronisation: the edge count stays on the device (row_ptr[N]) and every kernel bounds itself by it.
#include "common.cuh"

long long g_arreau_launches = 0;

namespace {

// ---- Philox4x32-10 counter-based generator (Salmon et al., SC'11) for throughput-run and evaluation noise ----
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
  const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
  const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
  c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
}
__device__ __forceinline__ void philox4x32_10(uint64_t seed, uint64_t ctr_lo, uint32_t ctr_hi, uint32_t stream_id,
                                              uint32_t (&out)[4]) {
  uint32_t c[4] = {(uint32_t)ctr_lo, (uint32_t)(ctr_lo >> 32), ctr_hi, stream_id};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) out[i] = c[i];
}
__device__ __forceinline__ double u01(uint32_t a, uint32_t b) {   // 53-bit uniform in [0,1)
  const uint64_t v = ((uint64_t)a << 21) ^ (uint64_t)(b >> 11);
  return (double)(v & ((1ull << 53) - 1)) * (1.0 / 9007199254740992.0);
}
// Box-Muller: two N(0,1) from one Philox output
__device__ __forceinline__ void box_muller(const uint32_t (&r)[4], double& v0, double& v1) {
  const double u1 = 1.0 - u01(r[0], r[1]), u2 = u01(r[2], r[3]);   // u1 in (0,1]
  const double rad = sqrt(-2.0 * log(u1));
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  v0 = rad * c;
  v1 = rad * s;
}

__global__ void step_noise_kernel(uint64_t seed, int step, long long n_normal, long long n_uniform,
                                  double* __restrict__ z_len, long long n_len, double* __restrict__ z_frac,
                                  double* __restrict__ u, const int32_t* __restrict__ step_ptr) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (step_ptr) step = *step_ptr;       // replayable step: the step ordinal of the current replay
  uint32_t r[4];
  if (idx < (n_normal + 1) / 2) {   // Box-Muller: two normals per counter
    philox4x32_10(seed, (uint64_t)idx, (uint32_t)step, 0u, r);
    const long long k0 = 2 * idx, k1 = 2 * idx + 1;
    double v0, v1;
    box_muller(r, v0, v1);
    if (k0 < n_len) z_len[k0] = v0; else z_frac[k0 - n_len] = v0;
    if (k1 < n_normal) {
      if (k1 < n_len) z_len[k1] = v1; else z_frac[k1 - n_len] = v1;
    }
  }
  if (idx < (n_uniform + 1) / 2) {
    philox4x32_10(seed, (uint64_t)idx, (uint32_t)step, 1u, r);
    u[2 * idx] = u01(r[0], r[1]);
    if (2 * idx + 1 < n_uniform) u[2 * idx + 1] = u01(r[2], r[3]);
  }
}

// Per-crystal keyed draws (arreau_eval_noise, arreau_sample_init_keyed, arreau_sample_noise_keyed).  Key = seed,
// counter = {crystal id (64 bits), index within the crystal, tag word}.  A step's draws carry the step ordinal above the
// tag's low 4 bits (tag | step << 4, step < 2^28), so no draw of a trajectory meets another, and the tags 2..10 keep
// every keyed draw apart from arreau_step_noise's tags 0 and 1.
struct KeyedTags {
  uint32_t cell;              // per crystal, counter 0: one uniform (the timestep or the initial angle), if drawn
  uint32_t len, len_ctr0;     // per crystal, counters len_ctr0, len_ctr0 + 1: three normals
  uint32_t frac;              // per atom a, counters 2a, 2a + 1: three normals
  uint32_t type;              // per atom a, counters a H .. a H + H - 1 with H = ceil(Z/2): Z uniforms
};
constexpr KeyedTags kEvalTags{2, 3, 0, 4, 5};        // t, eps_l, eps_x, u of an evaluation batch
constexpr KeyedTags kInitTags{6, 6, 1, 7, 0};        // angle, lengths, frac of a sampler's initial state (no types)
constexpr KeyedTags kStepTags{0, 8, 0, 9, 10};       // z_len, z_frac, u of one sampler step
constexpr int kMaxKeyedStep = (1 << 28) - 1;

// Work items: [0, G) one per crystal, [G, G + 2N) two per atom (the normals), then ceil(Z/2) per atom (the uniforms).
// The per-crystal uniform goes to t_crystal as U{1..T} or to angles as the monoclinic (90, U(90, 180), 90) in degrees
// (quirk B5), whichever is given.  step_ptr (replay): the step ordinal is read from the device.
__global__ void keyed_noise_kernel(uint64_t seed, KeyedTags tags, int step, const int32_t* __restrict__ step_ptr, int G,
                                   int N, int Z, const int64_t* __restrict__ crystal_id,
                                   const int32_t* __restrict__ atom_offset, const int32_t* __restrict__ crystal_of_atom,
                                   int T, int32_t* __restrict__ t_crystal, double* __restrict__ angles,
                                   double* __restrict__ lengths, double frac_scale, double* __restrict__ frac,
                                   double* __restrict__ u) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (step_ptr) step = *step_ptr;
  const uint32_t hi = (uint32_t)step << 4;
  const int H = (Z + 1) / 2;
  uint32_t r[4];
  if (idx < G) {
    const int g = (int)idx;
    const uint64_t id = (uint64_t)crystal_id[g];
    if (t_crystal || angles) {
      philox4x32_10(seed, id, 0u, tags.cell | hi, r);
      const double c = u01(r[0], r[1]);
      if (t_crystal) t_crystal[g] = min(1 + (int)(c * (double)T), T);
      if (angles) {
        angles[3 * (size_t)g + 0] = 90.0;
        angles[3 * (size_t)g + 1] = 90.0 + 90.0 * c;
        angles[3 * (size_t)g + 2] = 90.0;
      }
    }
    double v[4];
    philox4x32_10(seed, id, tags.len_ctr0, tags.len | hi, r);
    box_muller(r, v[0], v[1]);
    philox4x32_10(seed, id, tags.len_ctr0 + 1, tags.len | hi, r);
    box_muller(r, v[2], v[3]);
#pragma unroll
    for (int d = 0; d < 3; ++d) lengths[3 * (size_t)g + d] = v[d];
    return;
  }
  long long j = idx - G;
  if (j < 2LL * N) {
    const int b = (int)(j >> 1), k = (int)(j & 1), g = crystal_of_atom[b];
    const uint32_t a = (uint32_t)(b - atom_offset[g]);
    philox4x32_10(seed, (uint64_t)crystal_id[g], 2u * a + k, tags.frac | hi, r);
    double v0, v1;
    box_muller(r, v0, v1);
    frac[3 * (size_t)b + 2 * k] = v0 * frac_scale;
    if (k == 0) frac[3 * (size_t)b + 1] = v1 * frac_scale;
    return;
  }
  j -= 2LL * N;
  if (j < (long long)N * H) {
    const int b = (int)(j / H), k = (int)(j % H), g = crystal_of_atom[b];
    const uint32_t a = (uint32_t)(b - atom_offset[g]);
    philox4x32_10(seed, (uint64_t)crystal_id[g], a * (uint32_t)H + k, tags.type | hi, r);
    u[(size_t)b * Z + 2 * k] = u01(r[0], r[1]);
    if (2 * k + 1 < Z) u[(size_t)b * Z + 2 * k + 1] = u01(r[2], r[3]);
  }
}

// Replayable step (CUDA graph): the per-step scalars live in device memory and advance by themselves.  One block:
// k = *counter; t = max(t_first - k, 1); dyn = {t, VP posterior coefficients of t}; t_of_atom[:] = t; step_out = k;
// then *counter = k + 1.
__global__ void __launch_bounds__(1024)
step_advance_kernel(int32_t* __restrict__ counter, int t_first, const double* __restrict__ vp_table, int N,
                    int32_t* __restrict__ t_of_atom, double* __restrict__ dyn, int32_t* __restrict__ step_out) {
  const int k = *counter;
  const int t = max(t_first - k, 1);
  for (int i = threadIdx.x; i < N; i += blockDim.x) t_of_atom[i] = t;
  if (threadIdx.x < 4) dyn[1 + threadIdx.x] = vp_table[4 * (size_t)t + threadIdx.x];
  __syncthreads();
  if (threadIdx.x == 0) {
    dyn[0] = (double)t;
    *step_out = k;
    *counter = k + 1;
  }
}

}  // namespace

int arreau_vp_lattice_reverse_dyn(const double* lengths, const float* len0, const int32_t* atom_offset, const double* z,
                                  const double* dyn, int32_t G, const int32_t* known_crystal,
                                  const double* known_lengths, const float* vp_alpha_bars, double* lengths_out,
                                  void* stream);   // csrc/state.cu

extern "C" int arreau_abi_version(void) { return 1; }

extern "C" int arreau_model_dims(int* num_ori, int* hidden, int* basis, int* widening, int* layers) {
  if (num_ori) *num_ori = kO;
  if (hidden) *hidden = kC;
  if (basis) *basis = kD;
  if (widening) *widening = kW / kC;
  if (layers) *layers = kL;
  return ARREAU_OK;
}

extern "C" int64_t arreau_launch_count(void) { return (int64_t)g_arreau_launches; }

extern "C" int arreau_workspace_bytes(int32_t N, int32_t G, int64_t edge_capacity, int32_t precision, int32_t F, int32_t Z,
                                      arreau_workspace_sizes* o) {
  if (!o) return ARREAU_ERR_NULL;
  if (N < 0 || G < 0 || edge_capacity < 0 || F <= 0 || Z <= 0) return ARREAU_ERR_BAD_SHAPE;
  if (precision != ARREAU_PRECISION_FP32 && precision != ARREAU_PRECISION_FP16) return ARREAU_ERR_UNSUPPORTED;
  const bool fp16 = precision == ARREAU_PRECISION_FP16;
  const int64_t node = (int64_t)N * kO * kC, n = N, g = G, e = edge_capacity;
  o->h = node * 4;
  o->y = fp16 ? ((n * kO + 127) / 128) * 128 * kC * 2 : node * 4;            // fp16: 128-row UMMA tile images
  o->kernels = (int64_t)kL * e * kO * kC * (fp16 ? 2 : 4);
  o->acc = n * (Z + 6) * 4;
  o->x1 = node * 4;
  o->debug_per_layer = node * 4;
  o->pool = (fp16 && Z + 6 == 96) ? (int64_t)(kL + 1) * ((n + 15) / 16) * 4 * kC * 16 * 4 : 0;
  o->x = n * F * 4; o->vec = n * 12 * 4; o->logits = n * Z * 4; o->score = n * 3 * 4; o->len0 = g * 3 * 4;
  o->pos = n * 3 * 8; o->raw_count = n * 4; o->deg = n * 4; o->row_ptr = (n + 1) * 4; o->num_neighbors_image = g * 8;
  o->src = e * 4; o->dst = e * 4; o->cell = e; o->dist = e * 8; o->dir = e * 3 * 8;
  o->z_len = g * 3 * 8; o->z_frac = n * 3 * 8; o->u_type = n * Z * 8;
  return ARREAU_OK;
}

namespace {

int launch_step_noise(uint64_t seed, int step, const int32_t* step_ptr, int G, int N, int Z, double* z_len,
                      double* z_frac, double* u, cudaStream_t s) {
  const long long n_len = 3LL * G, n_normal = n_len + 3LL * N, n_uniform = (long long)N * Z;
  const long long work = ((n_normal > n_uniform ? n_normal : n_uniform) + 1) / 2;
  step_noise_kernel<<<(unsigned)((work + 255) / 256), 256, 0, s>>>(seed, step, n_normal, n_uniform, z_len, n_len, z_frac,
                                                                    u, step_ptr);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

int launch_keyed_noise(uint64_t seed, const KeyedTags& tags, int step, const int32_t* step_ptr, int G, int N, int Z,
                       const int64_t* crystal_id, const int32_t* atom_offset, const int32_t* crystal_of_atom, int T,
                       int32_t* t_crystal, double* angles, double* lengths, double frac_scale, double* frac, double* u,
                       cudaStream_t s) {
  const long long work = (long long)G + 2LL * N + (long long)N * ((Z + 1) / 2);
  keyed_noise_kernel<<<(unsigned)((work + 255) / 256), 256, 0, s>>>(seed, tags, step, step_ptr, G, N, Z, crystal_id,
                                                                     atom_offset, crystal_of_atom, T, t_crystal, angles,
                                                                     lengths, frac_scale, frac, u);
  CUDA_LAUNCH_CHECK();
  return ARREAU_OK;
}

}  // namespace

extern "C" int arreau_step_noise(uint64_t seed, int32_t step, int32_t G, int32_t N, int32_t Z, double* z_len,
                                 double* z_frac, double* u, void* stream) {
  if (G < 0 || N < 0 || Z <= 0) return ARREAU_ERR_BAD_SHAPE;
  if (G == 0 && N == 0) return ARREAU_OK;   // an empty batch is a no-op (its buffers may be NULL)
  if (!z_len || !z_frac || !u) return ARREAU_ERR_NULL;
  return launch_step_noise(seed, step, nullptr, G, N, Z, z_len, z_frac, u, (cudaStream_t)stream);
}

extern "C" int arreau_eval_noise(uint64_t seed, int32_t G, int32_t N, int32_t Z, int32_t num_steps,
                                 const int64_t* crystal_id, const int32_t* atom_offset, const int32_t* crystal_of_atom,
                                 int32_t* t_crystal, double* eps_x, double* u, double* eps_l, void* stream) {
  if (G < 0 || N < 0 || Z <= 1 || Z > 128 || num_steps <= 0) return ARREAU_ERR_BAD_SHAPE;
  if (G == 0) return ARREAU_OK;
  if (!crystal_id || !atom_offset || !t_crystal || !eps_l || (N > 0 && (!crystal_of_atom || !eps_x || !u)))
    return ARREAU_ERR_NULL;
  return launch_keyed_noise(seed, kEvalTags, 0, nullptr, G, N, Z, crystal_id, atom_offset, crystal_of_atom, num_steps,
                            t_crystal, nullptr, eps_l, 1.0, eps_x, u, (cudaStream_t)stream);
}

extern "C" int arreau_sample_init_keyed(uint64_t seed, int32_t G, int32_t N, const int64_t* crystal_id,
                                        const int32_t* atom_offset, const int32_t* crystal_of_atom,
                                        double pos_sigma_max, double* angles, double* lengths, double* frac,
                                        void* stream) {
  if (G < 0 || N < 0) return ARREAU_ERR_BAD_SHAPE;
  if (G == 0) return ARREAU_OK;
  if (!crystal_id || !atom_offset || !angles || !lengths || (N > 0 && (!crystal_of_atom || !frac)))
    return ARREAU_ERR_NULL;
  return launch_keyed_noise(seed, kInitTags, 0, nullptr, G, N, 0, crystal_id, atom_offset, crystal_of_atom, 0, nullptr,
                            angles, lengths, pos_sigma_max, frac, nullptr, (cudaStream_t)stream);
}

extern "C" int arreau_sample_noise_keyed(uint64_t seed, int32_t step, int32_t G, int32_t N, int32_t Z,
                                         const int64_t* crystal_id, const int32_t* atom_offset,
                                         const int32_t* crystal_of_atom, double* z_len, double* z_frac, double* u,
                                         void* stream) {
  if (G < 0 || N < 0 || Z <= 0 || step < 0 || step > kMaxKeyedStep) return ARREAU_ERR_BAD_SHAPE;
  if (G == 0) return ARREAU_OK;
  if (!crystal_id || !atom_offset || !z_len || (N > 0 && (!crystal_of_atom || !z_frac || !u))) return ARREAU_ERR_NULL;
  return launch_keyed_noise(seed, kStepTags, step, nullptr, G, N, Z, crystal_id, atom_offset, crystal_of_atom, 0, nullptr,
                            nullptr, z_len, 1.0, z_frac, u, (cudaStream_t)stream);
}

#define ARREAU_TRY(call)        \
  do {                          \
    const int rc__ = (call);    \
    if (rc__ != ARREAU_OK) return rc__; \
  } while (0)

extern "C" int arreau_ponita_forward(const arreau_weights* w, const arreau_workspace* ws, int32_t precision,
                                     const float* x, const float* vec, const int32_t* row_ptr, const int32_t* src,
                                     const double* dist, const double* dir, const double* lattice,
                                     const int32_t* atom_offset, const int32_t* crystal_of_atom, int32_t N, int32_t G,
                                     double radius, float* logits, float* score, float* len0, void* stream) {
  if (!w || !ws) return ARREAU_ERR_NULL;
  if (N < 0 || G < 0) return ARREAU_ERR_BAD_SHAPE;
  if (N == 0) return ARREAU_OK;
  if (!row_ptr || !ws->h || !ws->y || !ws->acc || !ws->x1 || (ws->edge_capacity > 0 && !ws->kernels)) return ARREAU_ERR_NULL;
  if (precision != ARREAU_PRECISION_FP32 && precision != ARREAU_PRECISION_FP16) return ARREAU_ERR_UNSUPPORTED;
  const bool fp16 = precision == ARREAU_PRECISION_FP16;
  const int Z = w->num_states;
  const size_t node_elems = (size_t)N * kO * kC;
  cudaStream_t s = (cudaStream_t)stream;
  // fp16 tensor path with a pool buffer: the read-outs run on orientation-pooled features that the embedding and the
  // MLP epilogues keep up to date, so h is never re-read for them (one pooled read-out launch instead of L passes)
  // (the pooled kernels are specialised on Z + 6 == 96 columns; other z_tables use the per-layer read-out)
  float* const pool = (fp16 && w->readout_v && w->readout_bias && Z + 6 == 96) ? ws->pool : nullptr;
  const size_t pool_elems = (size_t)((N + 15) / 16) * 4 * kC * 16;   // one entry: [groups of 16 atoms][4][C][16]
  if (pool)
    ARREAU_TRY(arreau_node_embed_pooled(x, ws->onehot_types, Z, vec, w->w_embed_t, w->ori, N, w->num_scalar, w->num_vec,
                                        ws->h, pool, w->readout_v, stream));
  else if (ws->onehot_types)
    ARREAU_TRY(arreau_node_embed_typed(x, ws->onehot_types, Z, vec, w->w_embed_t, w->ori, N, w->num_scalar, w->num_vec,
                                       ws->h, stream));
  else
    ARREAU_TRY(arreau_node_embed(x, vec, w->w_embed_t, w->ori, N, w->num_scalar, w->num_vec, ws->h, stream));
  if (ws->h_debug) {
    cudaError_t e = cudaMemcpyAsync(ws->h_debug, ws->h, node_elems * sizeof(float), cudaMemcpyDeviceToDevice, s);
    if (e != cudaSuccess) return (int)e;
  }
  const int32_t* num_edges_ptr = row_ptr + N;
  if (fp16)
    ARREAU_TRY(arreau_edge_kernels_f16(dir, dist, lattice, crystal_of_atom, src, num_edges_ptr, ws->edge_capacity,
                                        w->ori, w->edge_w1_img, w->edge_w_img, w->b2, radius, ws->kernels, stream));
  else
    ARREAU_TRY(arreau_edge_kernels_f32(dir, dist, lattice, crystal_of_atom, src, num_edges_ptr, ws->edge_capacity,
                                       w->ori, w->w1m_t, w->w2_t, w->b2, w->wk_t, radius, (float*)ws->kernels,
                                       stream));
  const size_t layer_elems = (size_t)ws->edge_capacity * kO * kC;
  for (int l = 0; l < kL; ++l) {
    const void* kern = fp16 ? (const void*)((const uint16_t*)ws->kernels + (size_t)l * layer_elems)
                            : (const void*)((const float*)ws->kernels + (size_t)l * layer_elems);
    // long rows (uncapped graphs, E/N ~ 30..90): the fused kernel's one-warp-per-atom gather serialises a row's
    // edges 8 at a time; the CTA-per-atom gather + separate tensor-core fiber conv is faster there (C2 uncapped:
    // 22.3 ms of message pass per step fused against ~15 ms for the pair)
    const bool long_rows = fp16 && w->fiber_frag && ws->edge_capacity > 16LL * N;
    if (long_rows) {
      const void* frag = (const uint8_t*)w->fiber_frag + (size_t)l * kC * 32 * 16;
      ARREAU_TRY(arreau_message_gather(kern, 1, ws->h, row_ptr, src, N, 1, ws->x1, stream));
      ARREAU_TRY(arreau_fiber_norm(ws->x1, 1, w->fiber_kernel + (size_t)l * kO * kO * kC, frag, w->conv_bias + l * kC,
                                   w->ln_w + l * kC, w->ln_b + l * kC, N, ws->y, 1,
                                   ws->x2_debug ? ws->x2_debug + l * node_elems : nullptr, stream));
    } else
    ARREAU_TRY(arreau_message_fiber_norm(kern, fp16, ws->h, row_ptr, src, w->fiber_kernel + (size_t)l * kO * kO * kC,
                                         w->fiber_frag ? (const uint8_t*)w->fiber_frag + (size_t)l * kC * 32 * 16 : nullptr,
                                         w->conv_bias + l * kC, w->ln_w + l * kC, w->ln_b + l * kC, N, ws->y, fp16,
                                         ws->x1_debug ? ws->x1_debug + l * node_elems : ws->x1,
                                         ws->x2_debug ? ws->x2_debug + l * node_elems : nullptr, stream));
    if (pool)
      ARREAU_TRY(arreau_convnext_mlp_f16_pooled(ws->y, (const uint8_t*)w->mlp_w_img + (size_t)l * 8 * 32768,
                                                 w->mlp_b1 + l * kW, w->mlp_b2 + l * kC, w->layer_scale + l * kC,
                                                 (int64_t)N * kO, ws->h, w->ori, pool + (size_t)(l + 1) * pool_elems,
                                                 w->readout_v + (size_t)(l + 1) * kC * (Z + 6), Z, stream));
    else if (fp16)
      ARREAU_TRY(arreau_convnext_mlp_f16(ws->y, (const uint8_t*)w->mlp_w_img + (size_t)l * 8 * 32768,
                                          w->mlp_b1 + l * kW, w->mlp_b2 + l * kC, w->layer_scale + l * kC,
                                          (int64_t)N * kO, ws->h, stream));
    else
      ARREAU_TRY(arreau_convnext_mlp_f32((const float*)ws->y, w->mlp_w1_t + (size_t)l * kC * kW, w->mlp_b1 + l * kW,
                                         w->mlp_w2_t + (size_t)l * kW * kC, w->mlp_b2 + l * kC,
                                         w->layer_scale + l * kC, (int64_t)N * kO, ws->h, stream));
    if (ws->h_debug) {
      cudaError_t e = cudaMemcpyAsync(ws->h_debug + (size_t)(l + 1) * node_elems, ws->h, node_elems * sizeof(float),
                                      cudaMemcpyDeviceToDevice, s);
      if (e != cudaSuccess) return (int)e;
    }
    if (!pool)
      ARREAU_TRY(arreau_readout_accumulate(ws->h, w->wr_t + (size_t)l * kC * (Z + 4), w->br + l * (Z + 4), w->ori, N, Z,
                                           l == 0, ws->acc, stream));
  }
  if (pool) ARREAU_TRY(arreau_readout_pooled(pool, w->readout_v, w->readout_bias, N, Z, kL + 1, ws->acc, stream));
  ARREAU_TRY(arreau_readout_finalize(ws->acc, atom_offset, N, G, Z, pool ? 1 : kL, logits, score, len0, stream));
  return ARREAU_OK;
}

namespace {

int lattice_from_angles(const arreau_step_args* a, int G, void* stream) {
  if (a->angle_trig) return arreau_lattice_from_trig(a->lengths, a->angle_trig, G, a->lattice, stream);
  return arreau_lattice_from_params(a->lengths, a->angles, G, a->lattice, stream);
}

// The launches of one denoise step after its noise is in place.  The timestep is a->t with the VP coefficients of `a`,
// or, with t_of_atom, on the device: t_of_atom[N] and dyn = {t, VP coefficients} (arreau_denoise_step_replay).
int denoise_step_body(const arreau_weights* w, const arreau_workspace* ws, const arreau_step_args* a,
                      const int32_t* t_of_atom, const double* dyn, void* stream) {
  const int N = a->num_atoms_total, G = a->num_crystals, Z = w->num_states;
  const int t = t_of_atom ? 0 : a->t;
  // predict_scores: lattice, features, cartesian positions, graph, network   (diffusion_loss.py:112-197)
  ARREAU_TRY(lattice_from_angles(a, G, stream));
  ARREAU_TRY(arreau_assemble_features(a->frac, a->types, a->lengths, a->angles, a->lattice, a->atom_offset,
                                      a->crystal_of_atom, t_of_atom, t, a->vp_betas, a->fourier_w, a->emb, N, G, Z,
                                      a->x, a->vec, stream));
  ARREAU_TRY(arreau_frac_to_cart(a->frac, a->lattice, a->crystal_of_atom, N, a->pos, stream));
  const double r2 = a->radius * a->radius;
  ARREAU_TRY(arreau_graph_count(a->pos, a->lattice, a->atom_offset, a->crystal_of_atom, N, G, r2, a->cap, 1,
                                a->raw_count, a->deg, a->num_neighbors_image, stream));
  ARREAU_TRY(arreau_graph_scan(a->deg, a->row_ptr, N, stream));
  ARREAU_TRY(arreau_graph_fill(a->pos, a->lattice, a->atom_offset, a->crystal_of_atom, N, G, r2, a->cap, 1,
                               a->raw_count, a->row_ptr, ws->edge_capacity, a->src, a->dst, a->cell, a->dist, a->dir,
                               nullptr, nullptr, a->overflow_flag, stream));
  ARREAU_TRY(arreau_ponita_forward(w, ws, a->precision, a->x, a->vec, a->row_ptr, a->src, a->dist, a->dir, a->lattice,
                                   a->atom_offset, a->crystal_of_atom, N, G, a->radius, a->logits, a->score, a->len0,
                                   stream));
  // update: lengths, lattice, fractional coordinates, atom types   (diffusion_loss.py:338-349); the known part of the
  // state, if any, is overwritten inside the same kernels, so the lattice below is formed from the known lengths
  if (dyn)
    ARREAU_TRY(arreau_vp_lattice_reverse_dyn(a->lengths, a->len0, a->atom_offset, a->z_len, dyn, G, a->known_crystal,
                                             a->known_lengths, a->vp_alpha_bars, a->lengths, stream));
  else if (a->known_crystal)
    ARREAU_TRY(arreau_vp_lattice_reverse_known(a->lengths, a->len0, a->atom_offset, a->z_len, a->t, a->vp_cx0,
                                               a->vp_cxt, a->vp_denom, a->vp_var, G, a->known_crystal, a->known_lengths,
                                               a->vp_alpha_bars, a->lengths, stream));
  else
    ARREAU_TRY(arreau_vp_lattice_reverse(a->lengths, a->len0, a->atom_offset, a->z_len, a->t, a->vp_cx0, a->vp_cxt,
                                         a->vp_denom, a->vp_var, G, a->lengths, stream));
  ARREAU_TRY(lattice_from_angles(a, G, stream));
  if (a->known_atom)
    ARREAU_TRY(arreau_ve_pbc_reverse_known(a->frac, a->score, a->z_frac, t_of_atom, t, a->ve_sigmas, N, a->known_atom,
                                           a->known_frac, a->frac, stream));
  else
    ARREAU_TRY(arreau_ve_pbc_reverse(a->frac, a->score, a->z_frac, t_of_atom, t, a->ve_sigmas, N, a->frac, stream));
  if (a->update_types && a->known_atom)
    ARREAU_TRY(arreau_d3pm_reverse_known(a->types, a->logits, a->u_type, t_of_atom, t, a->q_keep, a->q_to_mask,
                                         a->onestep_keep, a->onestep_to_mask, a->num_steps, N, Z, a->crystal_of_atom,
                                         a->allowed_states, a->known_atom, a->types, stream));
  else if (a->update_types && a->allowed_states)
    ARREAU_TRY(arreau_d3pm_reverse_allowed(a->types, a->logits, a->u_type, t_of_atom, t, a->q_keep, a->q_to_mask,
                                           a->onestep_keep, a->onestep_to_mask, a->num_steps, N, Z, a->crystal_of_atom,
                                           a->allowed_states, a->types, stream));
  else if (a->update_types)
    ARREAU_TRY(arreau_d3pm_reverse(a->types, a->logits, a->u_type, t_of_atom, t, a->q_keep, a->q_to_mask,
                                   a->onestep_keep, a->onestep_to_mask, a->num_steps, N, Z, a->types, stream));
  return ARREAU_OK;
}

}  // namespace

extern "C" int arreau_denoise_step(const arreau_weights* w, const arreau_workspace* ws, const arreau_step_args* a,
                                   void* stream) {
  if (!w || !ws || !a) return ARREAU_ERR_NULL;
  const int N = a->num_atoms_total, G = a->num_crystals, Z = w->num_states;
  if (N < 0 || G < 0) return ARREAU_ERR_BAD_SHAPE;
  if (N == 0 || G == 0) return ARREAU_OK;
  if (w->num_scalar != Z + 2 * a->emb + 10 || w->num_vec != 4) return ARREAU_ERR_BAD_SHAPE;
  return denoise_step_body(w, ws, a, nullptr, nullptr, stream);
}

// The same step with every per-step scalar in device memory, so that ONE captured CUDA graph replays the whole
// trajectory: replay k runs timestep t = max(t_first - k, 1) with Philox noise of step ordinal k (bit-identical to
// arreau_step_noise(seed, k) + arreau_denoise_step(t), or with r->crystal_id to arreau_sample_noise_keyed(seed, k)).
// capped graphs only (no host read of the edge count).
extern "C" int arreau_denoise_step_replay(const arreau_weights* w, const arreau_workspace* ws, const arreau_step_args* a,
                                          const arreau_step_replay* r, void* stream) {
  if (!w || !ws || !a || !r) return ARREAU_ERR_NULL;
  if (!r->counter || !r->vp_table || !r->t_of_atom || !r->dyn || !r->step_out) return ARREAU_ERR_NULL;
  const int N = a->num_atoms_total, G = a->num_crystals, Z = w->num_states;
  if (N < 0 || G < 0) return ARREAU_ERR_BAD_SHAPE;
  if (a->cap <= 0) return ARREAU_ERR_UNSUPPORTED;
  if (N == 0 || G == 0) return ARREAU_OK;
  if (w->num_scalar != Z + 2 * a->emb + 10 || w->num_vec != 4) return ARREAU_ERR_BAD_SHAPE;
  cudaStream_t s = (cudaStream_t)stream;
  step_advance_kernel<<<1, 1024, 0, s>>>(r->counter, r->t_first, r->vp_table, N, r->t_of_atom, r->dyn, r->step_out);
  CUDA_LAUNCH_CHECK();
  // (the step's noise buffers are inputs of arreau_denoise_step; here the call itself fills them)
  double* const z_len = const_cast<double*>(a->z_len);
  double* const z_frac = const_cast<double*>(a->z_frac);
  double* const u = const_cast<double*>(a->u_type);
  if (r->crystal_id)
    ARREAU_TRY(launch_keyed_noise(r->seed, kStepTags, 0, r->step_out, G, N, Z, r->crystal_id, a->atom_offset,
                                  a->crystal_of_atom, 0, nullptr, nullptr, z_len, 1.0, z_frac, u, s));
  else
    ARREAU_TRY(launch_step_noise(r->seed, 0, r->step_out, G, N, Z, z_len, z_frac, u, s));
  return denoise_step_body(w, ws, a, r->t_of_atom, r->dyn, stream);
}
