/*
 * arreau_b200 -- C ABI of the B200-native denoising step of the Arreau crystal diffusion model.
 *
 * The reference (curtischong/arreau) is pure Python/PyTorch and has no FFI layer: the drop-in
 * boundary is its Python module API (SURVEY.md section 8b), mirrored by the Python package
 * arreau_b200/.  Those Python mirrors reach the GPU ONLY through the entry points below
 * (ctypes, see arreau_b200/_lib.py and INTEGRATION.md).  Each entry point cites the reference
 * function it replaces (paths relative to the reference root).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer into caller-owned memory (torch tensors) unless it is one of
 *    the two plain-C argument structs (host memory, read during the call only); nothing is allocated
 *    or freed here; the caller sizes outputs and workspaces;
 *  - asynchronous on `stream` (a cudaStream_t passed as void*), no host synchronisation inside;
 *    the number of edges stays on the device (row_ptr[N]);
 *  - return 0 on success, a negative ARREAU_ERR_* for bad arguments, or the positive
 *    cudaError_t of a failed launch.  No exceptions, no aborts, no CPU fallback;
 *  - fp64 for geometry and diffusion state (the reference runs fp64), fp32 for the network
 *    (fp16 tensor-core operands with fp32 accumulation on the ARREAU_PRECISION_FP16 path);
 *  - the network kernels are specialised at compile time on the reference's default sizes
 *    (arreau_model_dims); any other size is ARREAU_ERR_UNSUPPORTED.
 */
#ifndef ARREAU_B200_H
#define ARREAU_B200_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ARREAU_OK 0
#define ARREAU_ERR_BAD_SHAPE (-1)
#define ARREAU_ERR_UNSUPPORTED (-2)
#define ARREAU_ERR_WORKSPACE (-3)
#define ARREAU_ERR_NULL (-4)

#define ARREAU_PRECISION_FP32 0 /* FFMA2 SIMT GEMMs, parity <= 1e-4 of the fp64 reference          */
#define ARREAU_PRECISION_FP16 1 /* tcgen05 fp16 operands, fp32 accumulate; tolerance stated in tests */
#define ARREAU_PRECISION_TF32 2 /* training backward only: TF32 tensor-core GEMMs, fp32 accumulate          */

/* Library/ABI version and the compile-time model dimensions (O=16, C=128, D=256, W=4, L=5). */
int arreau_abi_version(void);
int arreau_model_dims(int* num_ori, int* hidden, int* basis, int* widening, int* layers);
/* Number of kernels this library has launched since load (bench.py's gpu_launches). */
int64_t arreau_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * K1  periodic radius graph            replaces diffusion/diffusion_helpers.py:328-564
 *     (radius_graph_pbc, with SUPERCELLS :10).  Three launches so the caller can size E:
 *       count -> scan -> fill.   Edges come out receiver-major (i, then j, then cell 0..26),
 *       i.e. already CSR-by-receiver with row_ptr.
 * ------------------------------------------------------------------------------------------- */

/* Pass 1.  pos[N,3] f64 cartesian, lattice[G,3,3] f64 rows a,b,c, atom_offset[G+1] i32 (prefix
 * sum of num_atoms), crystal_of_atom[N] i32.  radius_sq = radius*radius evaluated by the caller
 * in double (helpers:432).  cap = max_num_neighbors_threshold (<= 0 disables, helpers:469-472).
 * LIMIT: cap <= 224 (the per-receiver selection buffer holds 256 candidates: cap + one 32-lane
 * batch); a larger positive cap returns ARREAU_ERR_UNSUPPORTED from both passes -- run uncapped
 * (cap <= 0) instead, which has no limit.  The reference's own configurations use 8 (Makefile:7).
 * Outputs: raw_count[N] i32 (bits 0..23: candidates with 1e-4 < d2 <= r2; bits 24..30: a scratch
 * hint for pass 2 -- the log-spaced distance bin that is known to contain the cap nearest; mask
 * with 0xFFFFFF to read the count), deg[N] i32 (= min(raw, cap) when cap > 0),
 * num_neighbors_image[G] i64 (helpers:456-465, incl. its cap<=0 quirk). */
int arreau_graph_count(const double* pos, const double* lattice, const int32_t* atom_offset,
                       const int32_t* crystal_of_atom, int32_t num_atoms_total, int32_t num_crystals,
                       double radius_sq, int32_t cap, int32_t remove_self_edges, int32_t* raw_count,
                       int32_t* deg, int64_t* num_neighbors_image, void* stream);

/* Exclusive scan deg[N] -> row_ptr[N+1] (row_ptr[N] = E stays on the device). */
int arreau_graph_scan(const int32_t* deg, int32_t* row_ptr, int32_t n, void* stream);

/* Pass 2.  Writes, for e in [row_ptr[i], row_ptr[i+1]): src[e] (sender j), dst[e] (= i),
 * cell[e] (index 0..26 into product((-1,0,1),repeat=3)), dist[e] f64, dir[e,3] f64
 * (= (pos_j + cell @ lattice) - pos_i, helpers:404-409,544).  Optional (may be NULL):
 * edge_index_i64[2,edge_capacity] (row 0 sender, row 1 receiver, row stride = edge_capacity)
 * and cell_offsets[E,3] f64 (= -cell, helpers:549).  Exact d2 ties under the cap are broken by
 * ascending (j, cell) -- torch.sort(stable=True) order.  Rows beyond edge_capacity are not
 * written and *overflow_flag (i32, may be NULL) is set to 1. */
int arreau_graph_fill(const double* pos, const double* lattice, const int32_t* atom_offset,
                      const int32_t* crystal_of_atom, int32_t num_atoms_total, int32_t num_crystals,
                      double radius_sq, int32_t cap, int32_t remove_self_edges, const int32_t* raw_count,
                      const int32_t* row_ptr, int64_t edge_capacity, int32_t* src, int32_t* dst,
                      int8_t* cell, double* dist, double* dir, int64_t* edge_index_i64,
                      double* cell_offsets, int32_t* overflow_flag, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K9  feature assembly                 replaces diffusion/diffusion_loss.py:124-158,
 *     diffusion/lattice_helpers.py:55-105 (lattice_from_params),
 *     diffusion/diffusion_helpers.py:23-25 (GaussianFourierProjection), :223-230 (frac_to_cart).
 * ------------------------------------------------------------------------------------------- */

/* lattice[G,3,3] f64 from lengths[G,3], angles[G,3] (radians as consumed by the reference). */
int arreau_lattice_from_params(const double* lengths, const double* angles, int32_t num_crystals,
                               double* lattice, void* stream);

/* Same, from per-crystal angle factors trig[G,6] = [sin b, cos b, sin a, cos g*, sin g*, cos a] that the caller
 * evaluated once (the angles are constant over a sampling trajectory): only the fp64 products of
 * lattice_helpers.py:85-96 are left, so the lattice is bit-identical to the reference's whatever libm the
 * factors came from. */
int arreau_lattice_from_trig(const double* lengths, const double* trig, int32_t num_crystals, double* lattice,
                             void* stream);

/* pos[N,3] = frac[N,3] @ lattice[crystal_of_atom] (f64). */
int arreau_frac_to_cart(const double* frac, const double* lattice, const int32_t* crystal_of_atom,
                        int32_t num_atoms_total, double* pos, void* stream);

/* Assemble the network inputs of predict_scores: x[N,F] f32 with F = Z + 2*emb + 10 laid out as
 * [onehot(types) | sin,cos(2 pi beta_t w) | n | lengths | angles | |lengths/n|] and
 * vec[N,4,3] f32 = [frac ; lattice rows].  The timestep of atom b is t_of_atom[b] (i32, may be
 * NULL -> every atom uses t); it indexes vp_betas[T+1] f64 (diffusion_loss.py:126).
 * fourier_w[emb] f64. */
int arreau_assemble_features(const double* frac, const int64_t* types, const double* lengths,
                             const double* angles, const double* lattice, const int32_t* atom_offset,
                             const int32_t* crystal_of_atom, const int32_t* t_of_atom, int32_t t,
                             const double* vp_betas, const double* fourier_w, int32_t emb,
                             int32_t num_atoms_total, int32_t num_crystals, int32_t num_states,
                             float* x, float* vec, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K2-K7  Ponita fiber-bundle forward   replaces ponita/models/ponita.py:88-155 and what it calls
 *     (ponita/nn/{conv,convnext,embedding}.py, ponita/transforms/*, ponita/geometry/invariants.py,
 *      ponita/utils/{to_from_sphere,windowing}.py, PyG add-aggregation and global_add_pool).
 *     Weight layouts are prepared by arreau_b200/weights.py.
 * ------------------------------------------------------------------------------------------- */

/* K3' (input independent): fiber_kernel[L,O,O,C] = fiber_kernel.weight_l @ fiber_basis_fn(ori.ori)
 * (ponita.py:66,95; conv.py:113).  w1[C,3] b1[C] w2[D,C] b2[D] wf[L,C,D], ori[O,3]. */
int arreau_fiber_kernel_precompute(const float* ori, const float* w1, const float* b1, const float* w2,
                                   const float* b2, const float* wf, float* fiber_kernel, void* stream);

/* K2: h0[N,O,C] = x_embedder([x | vec . ori_o]) (position_orientation_graph.py:84-86, ponita.py:98).
 * x[N,F] f32, vec[N,V,3] f32, w_embed_t[(F+V),C] f32 (transposed weight), ori[O,3]. */
int arreau_node_embed(const float* x, const float* vec, const float* w_embed_t, const float* ori,
                      int32_t num_atoms_total, int32_t num_scalar, int32_t num_vec, float* h, void* stream);

/* Same, when the first Z scalar features of x are a one-hot of types[N] (i64) as in predict_scores
 * (diffusion_loss.py:140-150): the one-hot block becomes one row lookup of the weight. */
int arreau_node_embed_typed(const float* x, const int64_t* types, int32_t num_states, const float* vec,
                            const float* w_embed_t, const float* ori, int32_t num_atoms_total, int32_t num_scalar,
                            int32_t num_vec, float* h, void* stream);

/* K3+K4a: per (edge, orientation) invariants -> 83 monomials -> Linear+GELU -> Linear+GELU -> *window
 * -> all L per-layer spatial kernels  kernels[L, edge_capacity, O, C] (ponita/geometry/invariants.py:17-22,
 * transforms/invariants.py:81-87, embedding.py:10-14, ponita.py:65,94, windowing.py:21-29,
 * conv.py:110).  dir[E,3]/dist[E] f64 from the graph; lattice[G,3,3] f64; crystal_of_atom[N];
 * src[E]; num_edges_ptr = &row_ptr[N] (device).  w1m_t[96,C]: rows 0..82 the monomial-folded first
 * layer, row 83 its bias, rows 84..95 zero; w2_t[C,D]; b2[D]; wk_t[D,L*C].
 * _f32: FFMA2 SIMT, fp32 kernels out.  _f16: tcgen05, fp16 operands, fp32 accumulation, fp16 kernels out;
 * its weights are UMMA tile images (K-major SWIZZLE_128B, arreau_b200/weights.py umma_tile_image):
 * w1_img = [128 x 128] image of w1m (32 KB, resident), w_img = 24 chunks of [128 x 64] (16 KB each):
 * W2 (n-half, k-slab) x 4, then for each layer the 4 k-slabs of conv.kernel.weight. */
int arreau_edge_kernels_f32(const double* dir, const double* dist, const double* lattice,
                            const int32_t* crystal_of_atom, const int32_t* src, const int32_t* num_edges_ptr,
                            int64_t edge_capacity, const float* ori, const float* w1m_t, const float* w2_t,
                            const float* b2, const float* wk_t, double radius, float* kernels, void* stream);
int arreau_edge_kernels_f16(const double* dir, const double* dist, const double* lattice,
                             const int32_t* crystal_of_atom, const int32_t* src, const int32_t* num_edges_ptr,
                             int64_t edge_capacity, const float* ori, const void* w1_img, const void* w_img,
                             const float* b2, double radius, void* kernels_f16, void* stream);

/* K4b+K5: x1[i,o,c] = sum_{e in row i} kernels[e,o,c] * h[src_e,o,c]   (conv.py:131-133 + PyG add)
 *         x2[i,p,c] = (1/O) sum_o x1[i,o,c] fiber_kernel[o,p,c] + bias[c]  (conv.py:115,126)
 *         y = LayerNorm_C(x2) * ln_w + ln_b                              (convnext.py:25)
 * `kernels` is ONE layer's [edge_capacity,O,C] slab (f32, or fp16 when kernels_f16 != 0);
 * fiber_kernel is that layer's [O,O,C].  y[N,O,C] is f32 row-major, or (y_f16) fp16 in 128-row UMMA tile
 * images for arreau_convnext_mlp_f16.  x1 ([N,O,C] f32 capacity, required) is the workspace between the two
 * launches (gather, then fiber conv + norm); it holds f32 [N,O,C] values, or -- when both kernels_f16 and y_f16 are set
 * (the fp16 tensor path, which also needs fiber_frag of this layer) -- f16 values transposed to [N,C,O]; x2_debug (f32 [N,O,C], may be NULL) receives x2 for the parity
 * tests.  Deterministic receiver-sorted CSR reduction (fixed order, no atomics). */
int arreau_message_fiber_norm(const void* kernels, int32_t kernels_f16, const float* h, const int32_t* row_ptr,
                              const int32_t* src, const float* fiber_kernel, const void* fiber_frag,
                              const float* conv_bias, const float* ln_w, const float* ln_b, int32_t num_atoms_total,
                              void* y, int32_t y_f16, float* x1, float* x2_debug, void* stream);

/* The two launches of arreau_message_fiber_norm as separate entry points (same arguments; used for per-kernel timing):
 * K4b gather: x1 = receiver-sorted CSR sums of kernels * h[src]; x1_f16_transposed != 0 (needs fp16 kernels) writes
 * fp16 x1t[N,C,O] instead of f32 x1[N,O,C].  K5: fiber conv + bias + LayerNorm of x1 -> y. */
int arreau_message_gather(const void* kernels, int32_t kernels_f16, const float* h, const int32_t* row_ptr,
                          const int32_t* src, int32_t num_atoms_total, int32_t x1_f16_transposed, float* x1,
                          void* stream);
int arreau_fiber_norm(const float* x1, int32_t x1_f16_transposed, const float* fiber_kernel, const void* fiber_frag,
                      const float* conv_bias, const float* ln_w, const float* ln_b, int32_t num_atoms_total, void* y,
                      int32_t y_f16, float* x2_debug, void* stream);

/* K4b+K5+LayerNorm of the fp16 tensor path as ONE launch (what arreau_message_fiber_norm runs when kernels_f16 and
 * y_f16 are both set): per 16-atom tile the receiver-sorted CSR sums are formed in shared memory (fp16, [atom][c][o]) and
 * consumed there by the tensor-core fiber conv + LayerNorm; x1 never goes to HBM.  Same arguments and results as the
 * gather + fiber_norm pair (bit-identical: same summation order, same roundings). */
int arreau_message_fiber_norm_fused(const void* kernels_f16, const float* h, const int32_t* row_ptr, const int32_t* src,
                                    const void* fiber_frag, const float* conv_bias, const float* ln_w,
                                    const float* ln_b, int32_t num_atoms_total, void* y_f16, float* x2_debug,
                                    void* stream);

/* fiber_frag[L][C][32] (16 bytes each): the fp16 mma.sync B fragments of fiber_kernel[L,O,O,C] / O, one per
 * (layer, channel, lane) -- the operand of the tensor-core fiber conv of the fp16 path (64 KB per layer). */
int arreau_fiber_frag_pack(const float* fiber_kernel, int32_t num_layers, void* fiber_frag, void* stream);

/* K6: h <- h + layer_scale * (W2 gelu(W1 y + b1) + b2)   (convnext.py:26-32); rows = N*O.
 * _f32: w1_t[C,4C], w2_t[4C,C] f32.  _f16: y_img = fp16 y as 128-row UMMA tile images (32 KB per tile, written
 * by arreau_message_fiber_norm with y_f16 != 0; ceil(rows/128) tiles must be allocated), w_img = 8 tile images
 * of 32 KB in issue order W1_0, W1_1, W2_0, W1_2, W2_1, W1_3, W2_2, W2_3 (128-wide slices of the hidden layer). */
int arreau_convnext_mlp_f32(const float* y, const float* w1_t, const float* b1, const float* w2_t,
                            const float* b2, const float* layer_scale, int64_t num_rows, float* h, void* stream);
int arreau_convnext_mlp_f16(const void* y_img, const void* w_img, const float* b1, const float* b2,
                             const float* layer_scale, int64_t num_rows, float* h, void* stream);

/* Pooled read-out path of the fp16 tensor path (K7 fused into K2 / K6; ponita.py:105-117, to_from_sphere.py:10-14).
 * The read-out Linear commutes with the orientation pooling, so only pooled features are needed, and the vector
 * channel only meets ONE weight row (row Z), so its contraction over the channels is done by the producer.
 * One pool ENTRY has a stride of ceil(N/16)*4*C*16 floats and holds
 *   [ceil(N/16)][C][16]       for each group of 16 atoms and channel c the 16 atoms' values of mean_o x[b,o,c],
 *   [ceil(N/16)*16][8]        per atom, element 2 d + half (d = 0..2; half = the producer's two channel halves):
 *                             sum_{c in half} V_k[c][Z] * (1/O) sum_o ori[o][d] x[b,o,c]
 * (the rest of the stride is unused).  pool is [L+1] entries: entry 0 pools the embedding output, entry k = 1..L pools
 * the residual UPDATE of interaction layer k (the feature after layer l is the sum of entries 0..l).
 * readout_v[L+1][C][Z+6], readout_bias[Z+6]: the per-entry sums of the read-out weights combined on the host
 * (arreau_b200/weights.py: pooled_readout_weights); readout_v_k = readout_v + k*C*(Z+6) is entry k's matrix.
 * arreau_node_embed_pooled: K2 that also writes entry 0 (types may be NULL).
 * arreau_convnext_mlp_f16_pooled: K6 whose two spare warps pool the residual update staged in shared memory into
 *   pool_out (one entry); h itself is updated as by arreau_convnext_mlp_f16.
 * arreau_readout_pooled: acc[N,Z+6] (column layout of arreau_readout_accumulate, already divided by L) =
 *   sum_k readout_v[k] pool[k] + readout_bias (fp32); entries = L+1. */
int arreau_node_embed_pooled(const float* x, const int64_t* types, int32_t num_states, const float* vec,
                             const float* w_embed_t, const float* ori, int32_t num_atoms_total, int32_t num_scalar,
                             int32_t num_vec, float* h, float* pool, const float* readout_v_0, void* stream);
int arreau_convnext_mlp_f16_pooled(const void* y_img, const void* w_img, const float* b1, const float* b2,
                                    const float* layer_scale, int64_t num_rows, float* h, const float* ori,
                                    float* pool_out, const float* readout_v_k, int32_t num_states, void* stream);
int arreau_readout_pooled(const float* pool, const float* readout_v, const float* readout_bias,
                          int32_t num_atoms_total, int32_t num_states, int32_t entries, float* acc, void* stream);

/* K7a: acc[N,Z+6] (+)= read-out of one layer pooled over orientations (ponita.py:105):
 *   acc[b, 0:Z]      mean_o (Wr h[b,o] + br)[0:Z]                (to_from_sphere.py:13-14)
 *   acc[b, Z:Z+3]    (1/O) sum_o (Wr h[b,o] + br)[Z] * ori_o      (to_from_sphere.py:10-11)
 *   acc[b, Z+3:Z+6]  mean_o (Wr h[b,o] + br)[Z+1:Z+4]
 * wr_t[C, Z+4] (transposed read-out weight), br[Z+4].  first_layer != 0 overwrites acc. */
int arreau_readout_accumulate(const float* h, const float* wr_t, const float* br, const float* ori,
                              int32_t num_atoms_total, int32_t num_states, int32_t first_layer, float* acc,
                              void* stream);

/* K7b: logits[N,Z], score[N,3] = acc / L; len0[G,3] = sum over atoms of crystal g of acc[.., Z+3:Z+6] / L
 * (ponita.py:108-117,152).  Fixed-order segment sum per crystal (deterministic). */
int arreau_readout_finalize(const float* acc, const int32_t* atom_offset, int32_t num_atoms_total,
                            int32_t num_crystals, int32_t num_states, int32_t num_layers, float* logits,
                            float* score, float* len0, void* stream);

/* All device weight pointers of one model (filled by arreau_b200/weights.py). */
typedef struct arreau_weights {
  const float* ori;          /* [O,3]                                                       */
  const float* w_embed_t;    /* [F+V, C]                                                    */
  const float* w1m_t;        /* [96, C]                                                     */
  const float* w2_t;         /* [C, D]                                                      */
  const float* b2;           /* [D]                                                         */
  const float* wk_t;         /* [D, L*C]                                                    */
  const float* fiber_kernel; /* [L,O,O,C]                                                   */
  const void* fiber_frag;    /* [L,C,32] x 16 B mma fragments of fiber_kernel / O (fp16 path), or NULL */
  const float* conv_bias;    /* [L,C]                                                       */
  const float* ln_w;         /* [L,C]                                                       */
  const float* ln_b;         /* [L,C]                                                       */
  const float* mlp_w1_t;     /* [L,C,4C]                                                    */
  const float* mlp_b1;       /* [L,4C]                                                      */
  const float* mlp_w2_t;     /* [L,4C,C]                                                    */
  const float* mlp_b2;       /* [L,C]                                                       */
  const float* layer_scale;  /* [L,C]                                                       */
  const float* wr_t;         /* [L,C,Z+4]                                                   */
  const float* br;           /* [L,Z+4]                                                     */
  /* fp16 operands of the tcgen05 path (NULL when only the fp32 path is used) */
  const void* edge_w1_img;   /* 32 KB UMMA tile image of w1m                                */
  const void* edge_w_img;    /* 24 x 16 KB UMMA tile images (W2, then Wk per layer)         */
  const void* mlp_w_img;     /* [L] x 8 x 32 KB UMMA tile images                            */
  const float* readout_v;    /* [L+1,C,Z+6] combined read-out matrices of the pooled read-out, or NULL */
  const float* readout_bias; /* [Z+6]                                                       */
  int32_t num_scalar;        /* F                                                           */
  int32_t num_vec;           /* V                                                           */
  int32_t num_states;        /* Z                                                           */
  int32_t reserved;
} arreau_weights;

/* Scratch of one forward pass, sized for num_atoms_total N and edge_capacity. */
typedef struct arreau_workspace {
  float* h;         /* [N,O,C] f32                                                           */
  void* y;          /* [N,O,C] f32 (fp32 path) or fp16 tile images, ceil(N*O/128)*32 KB (fp16 path) */
  void* kernels;    /* [L,edge_capacity,O,C] f32 or fp16                                     */
  float* acc;       /* [N,Z+6] f32                                                           */
  float* x1;        /* [N,O,C] f32: message sums between the gather and the fiber conv       */
  float* x1_debug;  /* NULL, or [L,N,O,C] f32                                                */
  float* x2_debug;  /* NULL, or [L,N,O,C] f32                                                */
  float* h_debug;   /* NULL, or [L+1,N,O,C] f32 (h after the embedding and after each layer) */
  int64_t edge_capacity;
  const int64_t* onehot_types; /* NULL, or types[N]: x[:, 0:Z] is one_hot(types) (lets the embedding skip the zeros) */
  float* pool;      /* NULL, or [L+1] pool entries (see arreau_readout_pooled) -> the fp16 path uses the pooled read-out */
} arreau_workspace;

/* Bytes of every buffer of arreau_workspace (and of the graph / step scratch of arreau_step_args) for N atoms, G
 * crystals, an edge capacity and a precision: what a caller allocates before arreau_ponita_forward /
 * arreau_denoise_step / arreau_denoise_step_replay (the caller owns all memory; nothing is allocated inside). */
typedef struct arreau_workspace_sizes {
  int64_t h, y, kernels, acc, x1, debug_per_layer, pool;          /* arreau_workspace (debug: x1/x2 take L, h L+1 layers) */
  int64_t x, vec, logits, score, len0;                            /* network io                                     */
  int64_t pos, raw_count, deg, row_ptr, num_neighbors_image;      /* graph scratch                                  */
  int64_t src, dst, cell, dist, dir;                              /* edge arrays                                    */
  int64_t z_len, z_frac, u_type;                                  /* noise                                          */
} arreau_workspace_sizes;
int arreau_workspace_bytes(int32_t num_atoms_total, int32_t num_crystals, int64_t edge_capacity, int32_t precision,
                           int32_t num_scalar, int32_t num_states, arreau_workspace_sizes* out);

/* PonitaFiberBundle.forward (ponita/models/ponita.py:88-123) on a prebuilt graph: x[N,F], vec[N,V,3] f32;
 * row_ptr[N+1], src[E] (receiver-sorted CSR), dist[E], dir[E,3] f64, lattice[G,3,3] f64.
 * Outputs logits[N,Z], score[N,3], len0[G,3] f32. */
int arreau_ponita_forward(const arreau_weights* w, const arreau_workspace* ws, int32_t precision, const float* x,
                          const float* vec, const int32_t* row_ptr, const int32_t* src, const double* dist,
                          const double* dir, const double* lattice, const int32_t* atom_offset,
                          const int32_t* crystal_of_atom, int32_t num_atoms_total, int32_t num_crystals,
                          double radius, float* logits, float* score, float* len0, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K8  per-step update                  replaces diffusion/diffusion_loss.py:338-349 with
 *     diffusion/diffusion_helpers.py:185-199 (VP_lattice.reverse_given_x0), :65-81 (VE_pbc.reverse),
 *     diffusion/d3pm.py:74-110,198-215 (D3PM.q_posterior_logits / reverse, mask chain).
 * ------------------------------------------------------------------------------------------- */

/* lengths'[G,3] = (cx0 * pred + cxt * lengths) / denom + var * z * [t>1]; the four coefficients are
 * evaluated by the caller with the reference's mixed fp32/fp64 arithmetic (quirk B1).
 * pred = len0[G,3] f32 * num_atoms (diffusion_loss.py:338). */
int arreau_vp_lattice_reverse(const double* lengths, const float* len0, const int32_t* atom_offset,
                              const double* z, int32_t t, double cx0, double cxt, double denom, double var,
                              int32_t num_crystals, double* lengths_out, void* stream);

/* frac'[N,3] = (frac - score*(s_t^2 - s_{t-1}^2) + sqrt(s_{t-1}^2 (s_t^2 - s_{t-1}^2)/s_t^2) z) mod 1
 * with torch.remainder semantics; t_of_atom may be NULL (then every atom uses t). */
int arreau_ve_pbc_reverse(const double* frac, const float* score, const double* z, const int32_t* t_of_atom,
                          int32_t t, const double* ve_sigmas, int32_t num_atoms_total, double* frac_out,
                          void* stream);

/* types'[N] = argmax(log(f1+eps) + log(f2+eps) + gumbel(u) * (0.2 + 0.8 [t != 1])), or logits if t == 1.
 * Mask-absorbing chain only (forward_type="mask", diffusion_loss.py:81): onestep_keep = 0.98,
 * onestep_to_mask = 0.02, q_keep[T], q_to_mask[T] = Qbar_t[0,0], Qbar_t[0,Z-1] (index t-1).
 * u[N,Z] f64 uniform noise. */
int arreau_d3pm_reverse(const int64_t* types, const float* logits, const double* u, const int32_t* t_of_atom,
                        int32_t t, const double* q_keep, const double* q_to_mask, double onestep_keep,
                        double onestep_to_mask, int32_t num_steps, int32_t num_atoms_total, int32_t num_states,
                        int64_t* types_out, void* stream);

/* The same step with the states restricted per crystal (chemical-system-constrained sampling).  allowed[G][4] u32:
 * bit d of allowed[4 g + d / 32] admits state d for the atoms of crystal g = crystal_of_atom[b] (bits at d >= Z are
 * ignored; a crystal with no bit below Z is unconstrained).  For an atom of crystal g with allowed set A:
 *   1. the x0 probabilities are the softmax of the logits over A; states outside A have probability 0 (this feeds
 *      sum_nomask, p_mask and f2);
 *   2. the candidates of the argmax are A plus the mask state Z-1 at t >= 2 (the absorbing state: a masked atom may stay
 *      masked) and A alone at t == 1.  States outside A are excluded explicitly: their posterior
 *      log(f1 + eps) + log(0 + eps) is finite, so the Gumbel noise could still select them;
 *   3. with every one of the Z bits set the output is bit-identical to arreau_d3pm_reverse.
 * A set without the mask bit ends every atom on an element of A.  Same checks and error codes as arreau_d3pm_reverse,
 * and ARREAU_ERR_NULL for a NULL crystal_of_atom or allowed (N > 0). */
int arreau_d3pm_reverse_allowed(const int64_t* types, const float* logits, const double* u, const int32_t* t_of_atom,
                                int32_t t, const double* q_keep, const double* q_to_mask, double onestep_keep,
                                double onestep_to_mask, int32_t num_steps, int32_t num_atoms_total, int32_t num_states,
                                const int32_t* crystal_of_atom, const uint32_t* allowed, int64_t* types_out,
                                void* stream);

/* Structure-conditioned sampling (RePaint replacement): the three reverse steps above with a known part of the state.
 * After the reverse update of timestep t, a known row is overwritten with a draw of the forward process at the new
 * level, q(x_{t-1} | x0), whose noise is the row's own step noise (its reverse draw is discarded, so no new draws):
 *   arreau_vp_lattice_reverse_known: a crystal g with known_crystal[g] != 0 gets
 *     lengths'[g] = sqrt(abar[t-1]) * known_lengths[g] + sqrt(1 - abar[t-1]) * z[g] at t >= 2 (vp_alpha_bars[T+1] f32,
 *     the arithmetic of arreau_vp_lattice_forward at level t-1: bit-identical), and known_lengths[g] at t == 1;
 *   arreau_ve_pbc_reverse_known: an atom b with known_atom[b] != 0 gets
 *     frac'[b] = (known_frac[b] + z[b] * ve_sigmas[t-1]) mod 1 at t >= 2 (arreau_ve_pbc_forward's frac_noisy at level
 *     t-1: bit-identical), and known_frac[b] (in [0,1)^3) at t == 1; t is the atom's t_of_atom[b] when given;
 *   arreau_d3pm_reverse_known: an atom with known_atom[b] != 0 keeps its state types[b] at every t; the others take
 *     arreau_d3pm_reverse's update, or arreau_d3pm_reverse_allowed's when allowed is given (crystal_of_atom then too;
 *     both may be NULL).
 * Every other row is bit-identical to the entry point without the suffix.  Same checks and error codes as those, and
 * ARREAU_ERR_NULL for a NULL known buffer or vp_alpha_bars (G, N > 0). */
int arreau_vp_lattice_reverse_known(const double* lengths, const float* len0, const int32_t* atom_offset,
                                    const double* z, int32_t t, double cx0, double cxt, double denom, double var,
                                    int32_t num_crystals, const int32_t* known_crystal, const double* known_lengths,
                                    const float* vp_alpha_bars, double* lengths_out, void* stream);
int arreau_ve_pbc_reverse_known(const double* frac, const float* score, const double* z, const int32_t* t_of_atom,
                                int32_t t, const double* ve_sigmas, int32_t num_atoms_total, const int32_t* known_atom,
                                const double* known_frac, double* frac_out, void* stream);
int arreau_d3pm_reverse_known(const int64_t* types, const float* logits, const double* u, const int32_t* t_of_atom,
                              int32_t t, const double* q_keep, const double* q_to_mask, double onestep_keep,
                              double onestep_to_mask, int32_t num_steps, int32_t num_atoms_total, int32_t num_states,
                              const int32_t* crystal_of_atom, const uint32_t* allowed, const int32_t* known_atom,
                              int64_t* types_out, void* stream);

/* Counter-based noise for throughput runs (the reference draws torch CPU noise, SURVEY 3.1): fills
 * z_len[G,3], z_frac[N,3] with N(0,1) and u[N,Z] with U[0,1) from Philox4x32-10 keyed by (seed, step). */
int arreau_step_noise(uint64_t seed, int32_t step, int32_t num_crystals, int32_t num_atoms_total,
                      int32_t num_states, double* z_len, double* z_frac, double* u, void* stream);

/* Per-crystal keyed sampling noise: the draws of DiffusionLoss.sample (diffusion_loss.py:294-301 initial state, :319-337
 * per-step noise) from Philox4x32-10 with key = seed and counter {c0, c1, c2, c3} = {crystal_id[g] (64 bits), index
 * within the crystal, tag word}, like arreau_eval_noise.  A crystal's draws -- and so its whole trajectory -- depend on
 * the seed, its id and its atom count only: not on its position in the batch, the batch's other crystals, the batch
 * size or the rank.  Same distributions as the reference's host draws, not the reference's torch / numpy CPU stream.
 * Tag words (disjoint from arreau_step_noise's 0, 1 and arreau_eval_noise's 2..5):
 *   6              initial cell: index 0 -> beta = 90 + 90 U[0,1) (angles (90, beta, 90), degrees consumed as radians,
 *                  quirk B5); indices 1, 2 -> lengths[3] N(0,1) (Box-Muller pairs, the 4th normal unused);
 *   7              initial frac: index 2a + k (atom a of the crystal, k = 0, 1) -> N(0,1) * pos_sigma_max;
 *   8 | step << 4  step noise z_len[3] (indices 0, 1, as tag 6's lengths);
 *   9 | step << 4  step noise z_frac (index 2a + k, as tag 7);
 *   10 | step << 4 step noise u[a, 2k .. 2k+1] (index a * ceil(Z/2) + k).
 * So the step ordinal is bounded by 0 <= step < 2^28 (ARREAU_ERR_BAD_SHAPE otherwise), and a crystal holds fewer than
 * 2^32 / ceil(Z/2) atoms.  crystal_id[G] i64, atom_offset[G+1], crystal_of_atom[N] of the batch.
 * arreau_sample_init_keyed writes angles[G,3], lengths[G,3], frac[N,3] (f64; frac is NOT wrapped, as the reference's);
 * arreau_sample_noise_keyed writes one step's z_len[G,3], z_frac[N,3] N(0,1) and u[N,Z] U[0,1) (f64). */
int arreau_sample_init_keyed(uint64_t seed, int32_t num_crystals, int32_t num_atoms_total, const int64_t* crystal_id,
                             const int32_t* atom_offset, const int32_t* crystal_of_atom, double pos_sigma_max,
                             double* angles, double* lengths, double* frac, void* stream);
int arreau_sample_noise_keyed(uint64_t seed, int32_t step, int32_t num_crystals, int32_t num_atoms_total,
                              int32_t num_states, const int64_t* crystal_id, const int32_t* atom_offset,
                              const int32_t* crystal_of_atom, double* z_len, double* z_frac, double* u, void* stream);

/* One whole denoise step (the body of the sampler loop, diffusion_loss.py:319-349), every kernel
 * above on one stream with no host synchronisation.  State is updated in place.
 * ABI note: allowed_states was appended after update_types, and the five known-state fields after allowed_states, so
 * the fields before them keep their offsets; a caller must zero-initialise them (or set them) -- a struct of an
 * earlier size is read past its end. */
typedef struct arreau_step_args {
  /* state, fp64 / i64, updated in place */
  double* frac;            /* [N,3]   */
  int64_t* types;          /* [N]     */
  double* lengths;         /* [G,3]   */
  const double* angles;    /* [G,3]   */
  const double* angle_trig;/* NULL, or [G,6] angle factors (see arreau_lattice_from_trig) */
  double* lattice;         /* [G,3,3] out: lattice_from_params(lengths', angles) */
  /* topology */
  const int32_t* atom_offset;      /* [G+1] */
  const int32_t* crystal_of_atom;  /* [N]   */
  int32_t num_atoms_total, num_crystals;
  /* graph scratch */
  double* pos;             /* [N,3]   */
  int32_t* raw_count;      /* [N]     */
  int32_t* deg;            /* [N]     */
  int32_t* row_ptr;        /* [N+1]   */
  int64_t* num_neighbors_image; /* [G] */
  int32_t* src;            /* [edge_capacity] */
  int32_t* dst;
  int8_t* cell;
  double* dist;
  double* dir;             /* [edge_capacity,3] */
  int32_t* overflow_flag;  /* [1] */
  /* network io */
  float* x;                /* [N,F]   */
  float* vec;              /* [N,4,3] */
  float* logits;           /* [N,Z]   */
  float* score;            /* [N,3]   */
  float* len0;             /* [G,3]   */
  /* noise (injected for parity runs, or filled by arreau_step_noise) */
  const double* z_len;     /* [G,3]   */
  const double* z_frac;    /* [N,3]   */
  const double* u_type;    /* [N,Z]   */
  /* tables */
  const double* vp_betas;  /* [T+1]   */
  const double* fourier_w; /* [emb]   */
  const double* ve_sigmas; /* [T+1]   */
  const double* q_keep;    /* [T]     */
  const double* q_to_mask; /* [T]     */
  double onestep_keep, onestep_to_mask;
  double vp_cx0, vp_cxt, vp_denom, vp_var;   /* coefficients of THIS timestep */
  int32_t emb, num_steps;  /* time-embedding half width (32), T */
  int32_t t;               /* timestep of this step (1..T-1) */
  int32_t cap;             /* max_neighbors */
  double radius;
  int32_t precision;
  int32_t update_types;    /* 0: keep types (constant_atoms mode, diffusion_loss.py:348-349) */
  const uint32_t* allowed_states; /* [G][4] device, or NULL (unconstrained): per-crystal allowed states of the type
                                     update (see arreau_d3pm_reverse_allowed) */
  /* structure conditioning (see arreau_ve_pbc_reverse_known): NULL known_atom / known_crystal = nothing known */
  const int32_t* known_atom;      /* [N] device, nonzero: the atom's position and type are known */
  const double* known_frac;       /* [N,3] its position in [0,1)^3 */
  const int32_t* known_crystal;   /* [G] device, nonzero: the crystal's lengths are known (its angles are a->angles) */
  const double* known_lengths;    /* [G,3] */
  const float* vp_alpha_bars;     /* [T+1] f32 abar table, needed with known_crystal */
} arreau_step_args;

int arreau_denoise_step(const arreau_weights* w, const arreau_workspace* ws, const arreau_step_args* a,
                        void* stream);

/* The same loop body (diffusion_loss.py:318-349 including the `for timestep in reversed(range(1, T))` bookkeeping)
 * with every per-step scalar in DEVICE memory, so that one captured CUDA graph of this call replays the whole
 * trajectory: replay k (k = *counter, incremented by the call) runs timestep t = max(t_first - k, 1) with Philox noise
 * of step ordinal k written into a->z_len / z_frac / u_type -- bit-identical to arreau_step_noise(seed, k, ...)
 * followed by arreau_denoise_step with a->t = t and the VP posterior coefficients of t.  a->t and a->vp_* are ignored.
 * With crystal_id set, the noise of replay k is arreau_sample_noise_keyed(seed, k, ..., crystal_id, ...) instead (the
 * per-crystal keyed draws; k < 2^28); NULL keeps the per-batch noise above, bit for bit.
 * Capped graphs only (max_neighbors > 0: no host read of the edge count); ARREAU_ERR_UNSUPPORTED otherwise.
 * ABI note: crystal_id was appended after `reserved`, so the fields before it keep their offsets; a caller must
 * zero-initialise it (or set it) -- a struct of the earlier size is read past its end. */
typedef struct arreau_step_replay {
  int32_t* counter;        /* [1] device: replays done so far; reset it to restart a trajectory */
  const double* vp_table;  /* [T+1][4] device: {cx0, cxt, denom, var} of VP_lattice.reverse_given_x0 per timestep */
  int32_t* t_of_atom;      /* [N] device scratch: the replay's timestep for the per-atom kernels */
  double* dyn;             /* [5] device scratch: {t, cx0, cxt, denom, var} of the replay */
  int32_t* step_out;       /* [1] device scratch: the replay's step ordinal (read by the noise kernel) */
  uint64_t seed;           /* Philox seed */
  int32_t t_first;         /* timestep of replay 0 (T - 1 for a whole trajectory) */
  int32_t reserved;
  const int64_t* crystal_id; /* [G] device, or NULL: per-crystal keyed noise (see arreau_sample_noise_keyed) */
} arreau_step_replay;

int arreau_denoise_step_replay(const arreau_weights* w, const arreau_workspace* ws, const arreau_step_args* a,
                               const arreau_step_replay* r, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Training step (SURVEY 8a rows a19-a23)   replaces DiffusionLoss.__call__ (diffusion/diffusion_loss.py:204-274),
 *     the forward noising it calls, and the autograd backward of the network (trainer.fit, main_diffusion.py:307).
 *     The forward pass of a training step is arreau_ponita_forward (fp32) run with ws->h_debug / x1_debug /
 *     x2_debug set, so that every layer's h, x1, x2 and the per-layer spatial kernels stay in memory.
 * ------------------------------------------------------------------------------------------- */

/* lengths[G,3], angles[G,3] (radians) of lattice[G,3,3]            (diffusion/lattice_helpers.py:16-35) */
int arreau_matrix_to_params(const double* lattice, int32_t num_crystals, double* lengths, double* angles, void* stream);

/* VE_pbc.forward (diffusion/diffusion_helpers.py:43-63): frac_noisy = (frac0 + eps * sigma_t) % 1 and the training
 * target = frac coordinates (% 1) of the minimum-image cartesian vector from the clean to the noisy position over the
 * 27 cells (min_distance_sqr_pbc :254-325, cart_to_frac_coords :233-251).  eps[N,3] is the injected randn. */
int arreau_ve_pbc_forward(const double* frac0, const double* eps, const int32_t* t_of_atom, const double* ve_sigmas,
                          const double* lattice, const int32_t* crystal_of_atom, int32_t num_atoms_total,
                          double* frac_noisy, double* target_eps, void* stream);

/* VP_lattice.forward (helpers:156-163): sqrt(abar_t) lengths + sqrt(1 - abar_t) eps with the fp32 abar table (B1). */
int arreau_vp_lattice_forward(const double* lengths, const double* eps, const int32_t* t_of_crystal,
                              const float* vp_alpha_bars, int32_t num_crystals, double* noisy_lengths, void* stream);

/* D3PM.get_xt / q_sample (diffusion/d3pm.py:119-127,139-143), mask chain: argmax(log(Qbar_t[x0,:] + eps) + gumbel(u)). */
int arreau_d3pm_q_sample(const int64_t* types0, const double* u, const int32_t* t_of_atom, const double* q_keep,
                         const double* q_to_mask, int32_t num_atoms_total, int32_t num_states, int64_t* types_t,
                         void* stream);

/* The three-term loss (diffusion_loss.py:95-110,253-274; d3pm.py:74-117,145-163) and its gradient with respect to
 * the network outputs.  loss_out[5] f64 = {loss, wrapped-MSE(frac), vb, ce, MSE(lengths / n)} with
 * loss = frac + (hybrid_coeff * vb + ce) + lattice.  terms_scratch: 3*N doubles.  Fixed-order reductions. */
int arreau_training_loss(const float* score, const float* logits, const float* len0, const double* target_eps,
                         const int64_t* types0, const int64_t* types_t, const int32_t* t_of_atom, const double* lengths,
                         const int32_t* atom_offset, const double* q_keep, const double* q_to_mask, double onestep_keep,
                         double onestep_to_mask, int32_t num_steps, int32_t num_atoms_total, int32_t num_crystals,
                         int32_t num_states, double hybrid_coeff, double* terms_scratch, double* loss_out, float* dscore,
                         float* dlogits, float* dlen0, void* stream);

/* ---- evaluation (validation / test loss) ---------------------------------------------------------------------- */

/* The random draws of DiffusionLoss.__call__ (diffusion_loss.py:213-216 timestep t ~ U{1..T}; :228-237 eps_x[N,3] ~ N(0,1),
 * u[N,Z] ~ U[0,1), eps_l[G,3] ~ N(0,1)), drawn PER CRYSTAL: Philox4x32-10 with key = seed and counter = {crystal_id[g]
 * (64 bits), index within the crystal, stream tag}.  A crystal's draws depend on the seed and its own id only -- not on
 * its position in the batch, the batch size or the rank -- so a loss evaluated with them does not depend on how a split
 * is grouped into batches or spread over GPUs.  Same distributions as the reference's draws, but not the reference's
 * torch CPU stream.  crystal_id[G] i64 (the crystal's index in its dataset), atom_offset[G+1], crystal_of_atom[N] of
 * the batch; outputs t_crystal[G] i32, eps_x[N,3], u[N,Z], eps_l[G,3] f64.  2 <= num_states <= 128. */
int arreau_eval_noise(uint64_t seed, int32_t num_crystals, int32_t num_atoms_total, int32_t num_states, int32_t num_steps,
                      const int64_t* crystal_id, const int32_t* atom_offset, const int32_t* crystal_of_atom,
                      int32_t* t_crystal, double* eps_x, double* u, double* eps_l, void* stream);

/* The loss of arreau_training_loss per crystal, without gradients (forward-only evaluation of
 * diffusion_loss.py:95-110,253-274; d3pm.py:74-117,145-163).  per_crystal[G][4] f64 = {sum of the wrapped squared frac
 * error, sum of vb, sum of ce over the crystal's atoms (in atom order), sum_d (len0 - lengths / n)^2}.  The per-atom
 * terms (terms_scratch, 3*N doubles: frac, vb, ce) come from the same device code as arreau_training_loss's.  A batch B's
 * loss_out is rebuilt from these sums: frac, vb, ce divided by N_B, the lattice term by 3 G_B,
 * loss = frac + (hybrid_coeff * vb + ce) + lattice.  2 <= num_states <= 128. */
int arreau_eval_loss(const float* score, const float* logits, const float* len0, const double* target_eps,
                     const int64_t* types0, const int64_t* types_t, const int32_t* t_of_atom, const double* lengths,
                     const int32_t* atom_offset, const double* q_keep, const double* q_to_mask, double onestep_keep,
                     double onestep_to_mask, int32_t num_steps, int32_t num_atoms_total, int32_t num_crystals,
                     int32_t num_states, double* terms_scratch, double* per_crystal, void* stream);

/* Flat parameter / gradient buffer: every trainable tensor of the reference's state_dict in its own layout
 * ([out, in] row-major), per-layer tensors stacked over the L layers, at these float offsets (SURVEY 8b names):
 * basis_fn.{1,3}.{weight,bias}, fiber_basis_fn.{1,3}.{weight,bias}, x_embedder.weight, then per layer
 * layer_scale, conv.bias, conv.kernel.weight, conv.fiber_kernel.weight, linear_1.{weight,bias},
 * linear_2.{weight,bias}, norm.{weight,bias}, read_out_layers.{weight,bias}. */
typedef struct arreau_train_layout_t {
  int64_t basis_w1, basis_b1, basis_w2, basis_b2, fiber_w1, fiber_b1, fiber_w2, fiber_b2, embed_w;
  int64_t layer_scale, conv_bias, conv_kernel_w, conv_fiber_w, lin1_w, lin1_b, lin2_w, lin2_b, norm_w, norm_b;
  int64_t readout_w, readout_b, total;
} arreau_train_layout_t;
int arreau_train_layout(int32_t num_scalar, int32_t num_vec, int32_t num_states, arreau_train_layout_t* layout);

/* Bytes of float workspace arreau_ponita_backward needs for N atoms and this edge capacity. */
int64_t arreau_ponita_backward_workspace_bytes(int32_t num_atoms_total, int64_t edge_capacity, int32_t num_scalar,
                                               int32_t num_vec);

/* Gradient of sum(dlogits*logits) + sum(dscore*score) + sum(dlen0*len0) with respect to every parameter (autograd
 * of ponita/models/ponita.py:88-155 and the layers it calls).  params / grads: flat buffers in arreau_train_layout_t
 * order (grads is overwritten).  w / ws: the packed weights and the workspace of the forward pass that produced the
 * outputs (ws->h_debug, x1_debug, x2_debug, kernels must hold that pass; fp32 path).  fold_table[258] i32: monomial
 * index of each PolynomialFeatures(3) column.  Deterministic: split reductions with a fixed-order second stage and a
 * sender-side gather for the transposed message pass, no atomics.  precision: ARREAU_PRECISION_FP32 (FFMA GEMMs,
 * the parity path) or ARREAU_PRECISION_TF32 (every GEMM of the backward on tcgen05 kind::tf32 tensor cores with fp32
 * accumulation in TMEM, operands fetched through TFLOAT32 tensor maps -- the TMA engine rounds them to 10 mantissa bits --
 * gradients within ~1e-3 of the fp32 path).
 * forward_kept: 0 after arreau_ponita_forward (the edge chain and the ConvNext hidden layers are recomputed here),
 * 1 after arreau_ponita_forward_train on the same `workspace` (they are read from it). */
int arreau_ponita_backward(const float* params, const arreau_train_layout_t* layout, const arreau_weights* w,
                           const arreau_workspace* ws, const int32_t* fold_table, const float* x, const float* vec,
                           const int32_t* row_ptr, const int32_t* src, const int32_t* dst, const double* dist,
                           const double* dir, const double* lattice, const int32_t* atom_offset,
                           const int32_t* crystal_of_atom, int32_t num_atoms_total, int32_t num_crystals, double radius,
                           const float* dlogits, const float* dscore, const float* dlen0, float* workspace,
                           int64_t workspace_bytes, float* grads, int32_t precision, int32_t forward_kept, void* stream);

/* The training forward with every dense contraction on the same generic GEMM as the backward (tcgen05 kind::tf32 under
 * ARREAU_PRECISION_TF32: the edge chain monomials -> basis MLP -> kernel basis, the five kernel projections and the
 * ConvNext MLP of every layer) and its activations KEPT in `workspace` (same layout and size as
 * arreau_ponita_backward's), so that arreau_ponita_backward(..., forward_kept = 1) does not recompute them.  Message
 * pass, fiber conv + LayerNorm, embedding and read-outs are the fp32 kernels of arreau_ponita_forward; ws must carry the
 * debug buffers (h / x1 / x2 of every layer) and fp32 `kernels`.  The node features of layer l are written straight into
 * slab l of ws->h_debug (ws->h itself is not touched).  Mathematics: ponita/models/ponita.py:88-123. */
int arreau_ponita_forward_train(const float* params, const arreau_train_layout_t* layout, const arreau_weights* w,
                                const arreau_workspace* ws, const int32_t* fold_table, const float* x, const float* vec,
                                const int32_t* row_ptr, const int32_t* src, const double* dist, const double* dir,
                                const double* lattice, const int32_t* atom_offset, const int32_t* crystal_of_atom,
                                int32_t num_atoms_total, int32_t num_crystals, double radius, float* workspace,
                                int64_t workspace_bytes, int32_t precision, float* logits, float* score, float* len0,
                                void* stream);

/* The fp32 GEMM the backward pass is built from: C[M,N] (=|+=) alpha * A * B (+ bias[n]).  a_k_contiguous: A is stored
 * [M][K] (else [K][M]); b_k_contiguous: B is stored [N][K] (else [K][N]).  Long reductions (K) are split over CTAs
 * into `partial` and summed in a fixed order.  Bit 1 of either flag (value 2 or 3) selects the TF32 tensor-core variant.
 * Exposed for the parity tests. */
int arreau_sgemm(int32_t a_k_contiguous, int32_t b_k_contiguous, const float* A, int64_t lda, const float* B, int64_t ldb,
                 float* C, int64_t ldc, int32_t M, int32_t N, int64_t K, float alpha, const float* bias,
                 int32_t accumulate, float* partial, int64_t partial_floats, void* stream);

/* w1m_t[96,C]: basis_fn.1.weight[C,258] with the columns of equal monomials summed (fixed order), row 83 = the bias,
 * rows 84..95 zero -- the first-layer operand of arreau_edge_kernels_f32 (embedding.py:10-14 has only 83 distinct
 * monomials).  Used to re-pack the weights on the device after every optimizer step. */
int arreau_fold_basis_w1(const float* w1, const float* b1, const int32_t* fold_table, float* w1m_t, void* stream);

/* out[2] f64 = {sum, sum of squares} of x[n] f32 (minus sub_cols[i % 128] when given): the statistics of
 * FiberBundleConv.callibrate (ponita/nn/conv.py:122-123,140-146).  scratch: 512 doubles. */
int arreau_moments(const float* x, const float* sub_cols, int64_t n, double* scratch, double* out, void* stream);

/* One torch.optim.Adam step on the flat buffers (lightning_wrappers/diffusion.py:161-210: L2 weight decay on the
 * elements whose decay_mask byte is set, i.e. the Linear weights) after the trainer's global-norm clip
 * (main_diffusion.py:297, gradient_clip_val = 0.5): coef = min(1, max_grad_norm / (sqrt(grad_moments[1]) + 1e-6)),
 * grad_moments = the {sum, sum of squares} arreau_moments wrote for the gradient buffer (device memory, so the step
 * does not synchronise; NULL or max_grad_norm <= 0 disables clipping).  step counts from 1.  ema[n] (NULL: none, and
 * the step's arithmetic is unchanged): the exponential moving average of the weights, updated in the same pass from the
 * post-step parameters as ema = ema_decay * ema + (1 - ema_decay) * params (the NeMo EMAOptimizer rule; the caller
 * initialises ema to the weights before the run's first step); 0 <= ema_decay <= 1. */
int arreau_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, const uint8_t* decay_mask,
                     int64_t n, double lr, double beta1, double beta2, double eps, double weight_decay, int64_t step,
                     double max_grad_norm, const double* grad_moments, float* ema, double ema_decay, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Beyond the reference: quality metrics of generated crystals.  The reference post-processes its
 * samples with pymatgen (CDVAE's structure validity); there are no reference lines to cite.
 * ------------------------------------------------------------------------------------------- */

#define ARREAU_METRICS_VALID 1           /* not degenerate and min_dist >= min_dist_threshold            */
#define ARREAU_METRICS_UNKNOWN_ELEMENT 2 /* some Z outside 0..max_z or with atomic_mass[Z] <= 0           */
#define ARREAU_METRICS_DEGENERATE 4      /* see arreau_crystal_metrics; min_dist is NaN                    */
#define ARREAU_METRICS_EXTENDED_SEARCH 8 /* the 27 images of the reduced cell did not prove the minimum    */

/* Per-crystal structure metrics.  frac[N,3] f64 and lattice[G,3,3] f64 rows a, b, c (pos = frac @ lattice, Angstrom),
 * atomic_numbers[N] i64, atom_offset[G+1] i32 (prefix sum of the atom counts), atomic_mass[max_z+1] f64: mass of
 * Z = 0..max_z in amu, <= 0 for an unknown element.  Outputs per crystal:
 *   volume[G]       |det lattice|, A^3;
 *   min_dist[G]     the exact minimum over distinct pairs i < j and every lattice translation of |pos_j - pos_i + t|
 *                   (+inf below 2 atoms); the basis is size-reduced and the 27 images are extended to the box that
 *                   provably holds the minimum when they cannot (metrics.cu derives the bound);
 *   density[G]      sum of masses (atom order) * 1.66053906660 / volume, g/cm^3, NaN with an unknown element;
 *   num_elements[G] number of distinct known Z;
 *   flags[G]        ARREAU_METRICS_* bits.  VALID follows CDVAE: min_dist >= min_dist_threshold (0.5 A) and
 *                   volume >= min_volume (0.1 A^3).
 * A crystal is DEGENERATE (no search, min_dist NaN, not VALID) when a lattice entry or coordinate is not finite, its
 * volume is below min_volume, its atom_offset entries are out of order or outside 0..N, or the exact search would need
 * more than 16 images either way along an axis of the reduced cell (a cell height below 1/16 of the crystal's
 * shortest 27-image distance).  Any atom count is supported; one warp per crystal.  A crystal's outputs depend only
 * on that crystal, bit for bit, whatever batch it is in. */
int arreau_crystal_metrics(const double* frac, const double* lattice, const int64_t* atomic_numbers,
                           const int32_t* atom_offset, int32_t num_atoms_total, int32_t num_crystals,
                           const double* atomic_mass, int32_t max_z, double min_dist_threshold, double min_volume,
                           double* volume, double* min_dist, double* density, int32_t* num_elements, int32_t* flags,
                           void* stream);

/* ---------------------------------------------------------------------------------------------
 * Beyond the reference: a paired structure matcher for crystal structure prediction (match rate and
 * RMSE, as CDVAE and DiffCSP report them with pymatgen's StructureMatcher).  No reference lines to cite.
 * ------------------------------------------------------------------------------------------- */

#define ARREAU_MATCH_MATCHED 1       /* a candidate with rms < stol exists                                   */
#define ARREAU_MATCH_COMPOSITION 2   /* the multisets of Z differ (atom counts included); not searched       */
#define ARREAU_MATCH_DEGENERATE 4    /* non-finite input, |det| < 0.1 A^3, an empty crystal, atoms not sorted */
                                     /* by Z, bad offsets, or a reduction that did not converge              */
#define ARREAU_MATCH_SEARCH_LIMIT 8  /* a length band held more than 128 lattice points, or the search box   */
                                     /* more than 255 steps along a basis vector; not scored                 */
#define ARREAU_MATCH_TOO_LARGE 16    /* more than 256 atoms; not searched                                    */

/* Crystal g of set 1 (generated) against crystal g of set 2 (source), for g < num_pairs, as pymatgen's
 * StructureMatcher(stol, ltol, angle_tol, scale=True, attempt_supercell=False, primitive_cell=False)
 * .get_rms_dist(crystal1, crystal2) computes it (DiffCSP: stol 0.5, ltol 0.3, angle_tol 10 degrees); csrc/match.cu
 * states the steps and the pymatgen function each mirrors.  Per set: frac[N,3] f64, lattice[G,3,3] f64 rows a, b, c,
 * z[N] i64 and offset[G+1] i32 (prefix sums of the atom counts); within each crystal the atoms must be sorted by Z.
 * Outputs per pair: rms[G] and max_dist[G], the normalised (by (n / V_avg)^(1/3)) rms and largest displacement of
 * the candidate with the smallest rms over every lattice mapping and translation (NaN when no candidate exists or
 * the pair was not searched); num_mappings[G], the lattice mappings found; flags[G], ARREAU_MATCH_* bits (at most
 * one of COMPOSITION, DEGENERATE, SEARCH_LIMIT, TOO_LARGE).  Up to 256 atoms per crystal, fp64, one warp per pair;
 * a pair's outputs depend only on that pair, bit for bit, whatever batch it is in.  stol, ltol and angle_tol must be
 * finite and positive (ARREAU_ERR_BAD_SHAPE). */
int arreau_structure_match(const double* frac1, const double* lattice1, const int64_t* z1, const int32_t* offset1,
                           const double* frac2, const double* lattice2, const int64_t* z2, const int32_t* offset2,
                           int32_t num_atoms1, int32_t num_atoms2, int32_t num_pairs, double stol, double ltol,
                           double angle_tol, double* rms, double* max_dist, int32_t* num_mappings, int32_t* flags,
                           void* stream);

/* Pair p is crystal index1[p] of set 1 against crystal index2[p] of set 2, for p < num_pairs, as pymatgen's
 * StructureMatcher(stol, ltol, angle_tol, scale=True, attempt_supercell=False, primitive_cell=False)
 * .fit(crystal1, crystal2) decides it (pymatgen's defaults: stol 0.3, ltol 0.2, angle_tol 5 degrees): the steps of
 * arreau_structure_match, with a candidate's value its largest normalised distance instead of its rms, and the search
 * stopped at the first candidate below stol in the enumeration order; crystal1's lattice is the one mapped.  Per set:
 * frac, lattice, z and offset as above for num_crystals crystals and num_atoms atoms; index1[P], index2[P] i32.
 * Outputs per pair: max_dist[P], the first value below stol, else the smallest found (NaN when no candidate exists or
 * the pair was not searched); num_mappings[P], the lattice mappings visited (all of them when not matched); flags[P],
 * ARREAU_MATCH_* bits, MATCHED when fit holds, DEGENERATE also for an index outside its set.  The argument checks,
 * limits and determinism are those of arreau_structure_match. */
int arreau_structure_fit_pairs(const double* frac1, const double* lattice1, const int64_t* z1, const int32_t* offset1,
                               int32_t num_atoms1, int32_t num_crystals1, const double* frac2, const double* lattice2,
                               const int64_t* z2, const int32_t* offset2, int32_t num_atoms2, int32_t num_crystals2,
                               const int32_t* index1, const int32_t* index2, int32_t num_pairs, double stol,
                               double ltol, double angle_tol, double* max_dist, int32_t* num_mappings, int32_t* flags,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ARREAU_B200_H */
