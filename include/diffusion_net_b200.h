/*
 * diffusion_net_b200 -- C ABI of the B200-native DiffusionNetBlock hot path.
 *
 * The reference (nmwsharp/diffusion-net) is pure Python and has no FFI layer; its
 * boundary is the module API of src/diffusion_net/layers.py plus the operator
 * tuple of geometry.get_operators (SURVEY.md section 8b).  Each entry point below
 * replaces one reference function on that path and is what a reference-side ctypes
 * binding would call (INTEGRATION.md shows the stub).  Conventions:
 *
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless a
 *     name ends in _host; all float data is fp32, row-major, densely packed unless
 *     a leading dimension is given;
 *   - the caller allocates every output and the workspace (dn_workspace_bytes);
 *   - kernels are enqueued on `stream` (a cudaStream_t) and never synchronise;
 *   - return 0 on success, <0 for a DN_ERR_* argument/support error, >0 for a
 *     cudaError_t raised at launch; dn_error_string() explains either;
 *   - no global mutable state: calls on different streams are independent.
 *
 * `engine` selects the arithmetic of the dense contractions:
 *   DN_ENGINE_SIMT  exact fp32 FFMA (debug / gold-on-device, any shape)
 *   DN_ENGINE_TC3X  tcgen05 tensor cores, error-compensated 3xTF32 (fp32-grade,
 *                   the default product path; <=1e-5 relative vs the reference)
 *   DN_ENGINE_TC1X  tcgen05 single-pass TF32 (fast, ~5e-4 relative)
 *   DN_ENGINE_BF16  tcgen05 single-pass bf16 (kind::f16, fp32 accumulate; ~1e-2 relative; layers up to
 *                   256 wide chain on chip: BASELINE config 3, C_width = 256).  Tensors stay fp32 in HBM.
 */
#ifndef DIFFUSION_NET_B200_H
#define DIFFUSION_NET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DN_ABI_VERSION 5

typedef void* dn_stream_t; /* cudaStream_t */

enum dn_status {
  DN_OK = 0,
  DN_ERR_INVALID_ARGUMENT = -1, /* null pointer, negative size, mismatched dims   */
  DN_ERR_UNSUPPORTED = -2,      /* shape/engine combination not implemented        */
  DN_ERR_WORKSPACE = -3,        /* workspace too small (see dn_workspace_bytes)    */
  DN_ERR_NOT_SM100 = -4         /* tensor-core engine requested on a non-sm_100 GPU */
};

enum dn_engine { DN_ENGINE_SIMT = 0, DN_ENGINE_TC3X = 1, DN_ENGINE_TC1X = 2, DN_ENGINE_BF16 = 3 };

/* Shared-pattern CSR form of the (gradX, gradY) pair.  The reference hands over two
 * coalesced COO tensors with identical, row-sorted sparsity (Re/Im of one complex
 * matrix, geometry.py:381-382; utils.py:50-55).  vals holds (gx, gy) interleaved. */
struct dn_patches;
typedef struct dn_csr {
  const int32_t* rowptr; /* V+1 */
  const int32_t* colidx; /* nnz */
  const float* vals;     /* 2*nnz: gx0, gy0, gx1, gy1, ... */
  int64_t nnz;
  const struct dn_patches* patches; /* optional (NULL): locality structure for the gather kernel, see below */
} dn_csr;

/* Optional locality structure over a dn_csr, built once per mesh (dn_patch_build, host side) for operators that
 * stay resident.  The rows are grouped into patches of graph-adjacent vertices; the fused gradient-features
 * kernel then stages the distinct neighbour rows of a patch in shared memory once (coalesced) and gathers from
 * there, instead of re-fetching every neighbour row through L1/L2 for every vertex that touches it.  Results are
 * bit-identical to the unpatched kernel (same entries, same order, same arithmetic).  The struct lives in host
 * memory like dn_csr; the arrays are device arrays. */
typedef struct dn_patches {
  int32_t n_patches;
  int32_t max_src;         /* largest number of distinct source rows of any patch (sizes the shared memory) */
  const int32_t* tgt_ptr;  /* n_patches+1: the rows of patch p are tgt[tgt_ptr[p] .. tgt_ptr[p+1])           */
  const int32_t* tgt;      /* V: row ids in patch order, every row exactly once                              */
  const int32_t* src_ptr;  /* n_patches+1                                                                    */
  const int32_t* src_rows; /* distinct column ids (= gathered rows) of each patch                            */
  const int32_t* ent_ptr;  /* V+1: the entries of row tgt[i] are [ent_ptr[i], ent_ptr[i+1]) of lcol / vals   */
  const uint8_t* lcol;     /* nnz: index into the patch's src_rows                                           */
  const float* vals;       /* 2*nnz: (gx, gy) in patch order                                                 */
} dn_patches;

/* Parameters of one DiffusionNetBlock, named as in the reference state_dict
 * (layers.py:38, 110-113, 150-155).  nn.Linear layout: weight[n_out][n_in]. */
typedef struct dn_block_params {
  float* diffusion_time;     /* (C)   in/out: overwritten with max(t, 1e-8), layers.py:48-49 */
  const float* A_re;         /* (C,C) gradient_features.A_re.weight, or .A.weight when !rotations */
  const float* A_im;         /* (C,C) gradient_features.A_im.weight, NULL when !rotations        */
  int with_gradient_features;
  int with_gradient_rotations;
  int n_mlp_layers;          /* number of Linear layers in the MiniMLP (reference default 3)      */
  const float* const* mlp_weight_host; /* host array [n_mlp_layers] of device pointers            */
  const float* const* mlp_bias_host;   /* host array [n_mlp_layers] of device pointers            */
  const int* mlp_dims_host;  /* host array [n_mlp_layers+1]: 3C (or 2C), hidden..., C             */
} dn_block_params;

int dn_abi_version(void);
const char* dn_error_string(int code);
/* sm count / compute capability (major*10+minor) / opt-in shared memory per block of `device`. */
int dn_device_query(int device, int* sm_count, int* cc, int64_t* smem_optin_bytes);

/* Number of kernels this library has launched so far in this process (monotonic; bench.py
 * differences it around the timed region). */
int64_t dn_kernel_launch_count(void);

/* Bytes of scratch any call below needs for (V, K, C); 256-byte aligned base required. */
int64_t dn_workspace_bytes(int64_t V, int K, int C);

/* Operator prep: row-sorted COO (int64 rows/cols as in utils.py:55) -> dn_csr arrays.
 * vy may be NULL (single matrix; gy written as 0). */
int dn_csr_from_coo(const int64_t* rows, const int64_t* cols, const float* vx, const float* vy,
                    int64_t nnz, int64_t V, int32_t* rowptr, int32_t* colidx, float* vals,
                    dn_stream_t stream);

/* HOST-side operator prep (every pointer here is a HOST pointer): greedy breadth-first clustering of the CSR
 * pattern into patches of at most max_targets rows whose distinct columns number at most max_src (<= 256).
 * Outputs (caller-allocated): tgt_ptr, src_ptr (V+1 each: worst case one patch per row), tgt (V), src_rows (nnz),
 * ent_ptr (V+1), lcol (nnz), perm (nnz: patch-order entry -> CSR entry, for permuting vals), max_src_out (1).
 * Returns the number of patches, or a negative DN_ERR_* (a row longer than max_src is DN_ERR_UNSUPPORTED). */
int64_t dn_patch_build(int64_t V, const int32_t* rowptr_host, const int32_t* colidx_host, int max_targets,
                       int max_src, int32_t* tgt_ptr_host, int32_t* tgt_host, int32_t* src_ptr_host,
                       int32_t* src_rows_host, int32_t* ent_ptr_host, uint8_t* lcol_host, int32_t* perm_host,
                       int32_t* max_src_out_host);

/* Operator prep from the reference's on-disk cache (geometry.py:548-568 stores gradX/gradY as scipy CSC; the
 * read side is geometry.py:494-519): a CSC matrix is the CSR of its transpose, so the cache arrays are `in`
 * verbatim and this call produces the forward CSR (columns sorted inside every row, deterministic).
 * `in` and the outputs describe square V x V matrices; workspace needs 4*V bytes. */
int dn_csr_transpose(const dn_csr* in, int64_t V, int32_t* rowptr_out, int32_t* colidx_out,
                     float* vals_out, void* workspace, int64_t ws_bytes, dn_stream_t stream);

/* geometry.py:600-628 compute_hks: out(V,S)[v,s] = sum_k exp(-evals[k]*scales[s]) * evecs(V,K)[v,k]^2. */
int dn_compute_hks(const float* evals, const float* evecs, const float* scales, int64_t V, int K,
                   int S, float* out, dn_stream_t stream);

/* geometry.py:572-583 to_basis: out(K,C) = basis(V,K)^T @ (values(V,C) * massvec(V)[:,None]).
 * massvec may be NULL (no weighting; used by the backward pass). */
int dn_to_basis(const float* values, const float* basis, const float* massvec, int64_t V, int K,
                int C, float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* geometry.py:586-598 from_basis (real branch): out(V,C) = basis(V,K) @ values(K,C).
 * row_scale (V) optional: out rows multiplied by it (mass, backward pass). */
int dn_from_basis(const float* values, const float* basis, const float* row_scale, int64_t V, int K,
                  int C, float* out, void* workspace, int64_t ws_bytes, int engine,
                  dn_stream_t stream);

/* layers.py:44-67 LearnedTimeDiffusion.forward, method='spectral'.
 * time (C) is clamped in place (layers.py:48-49).  x_spec_out (K,C) optional: the
 * un-scaled spectral coefficients, saved for the backward pass. */
int dn_learned_time_diffusion_fwd(const float* x, const float* mass, const float* evals,
                                  const float* evecs, float* time, int64_t V, int K, int C,
                                  float* x_diffuse, float* x_spec_out, void* workspace,
                                  int64_t ws_bytes, int engine, dn_stream_t stream);

/* Backward of the above w.r.t. x and time (mass/evals/evecs are data, SURVEY.md 8a).
 * grad_time (C) is ACCUMULATED into (+=).  */
int dn_learned_time_diffusion_bwd(const float* grad_out, const float* mass, const float* evals,
                                  const float* evecs, const float* time, const float* x_spec,
                                  int64_t V, int K, int C, float* grad_x, float* grad_time,
                                  void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* layers.py:216-223: out(V,C,2) with out[v,c,0] = (gradX @ x)[v,c], out[v,c,1] = (gradY @ x)[v,c]. */
int dn_grad_spmm(const dn_csr* grad, const float* x, int64_t V, int C, float* out,
                 dn_stream_t stream);

/* layers.py:117-130 SpatialGradientFeatures.forward on vectors(V,C,2) -> out(V,C). */
int dn_spatial_gradient_features_fwd(const float* vectors, const float* A_re, const float* A_im,
                                     int with_gradient_rotations, int64_t V, int C, float* out,
                                     void* workspace, int64_t ws_bytes, int engine,
                                     dn_stream_t stream);

/* layers.py:216-226 fused: features(V,C) = SpatialGradientFeatures(stack(gradX@x, gradY@x)).
 * The dense maps are applied before the sparse gradient (P = x A_re^T, Q = x A_im^T; the two
 * operators commute by linearity), so the (V,C,2) tensor is never materialised.
 * pq_out (V,2C) optional: P|Q saved for the backward pass (workspace used if NULL). */
int dn_gradient_features_fwd(const dn_csr* grad, const float* x_diffuse, const float* A_re,
                             const float* A_im, int with_gradient_rotations, int64_t V, int C,
                             float* features, float* pq_out, void* workspace, int64_t ws_bytes,
                             int engine, dn_stream_t stream);

/* Backward of dn_gradient_features_fwd.  grad_t is the CSR of the TRANSPOSED pattern
 * (same (gx,gy) values permuted).  grad_x is written; grad_A_re / grad_A_im are ACCUMULATED. */
int dn_gradient_features_bwd(const dn_csr* grad, const dn_csr* grad_t, const float* grad_features,
                             const float* x_diffuse, const float* pq, const float* features,
                             const float* A_re, const float* A_im, int with_gradient_rotations,
                             int64_t V, int C, float* grad_x, float* grad_A_re, float* grad_A_im,
                             void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* Generic fused affine chain over vertex rows (MiniMLP layers.py:133-164, first_lin/last_lin
 * layers.py:366,373, and the block's cat+MLP+skip layers.py:229-239):
 *   h_0 = concat_s src[s](V, width[s]);  h_{l+1} = act_l(h_l @ W_l^T + b_l) (* dropmask_l);
 *   out = h_L (+ residual).
 * ReLU after every layer but the last.  hidden_out[l] (optional, l < L-1) receives h_{l+1}
 * (post-activation, post-mask) for the backward pass; drop_mask[l] (optional) is a (V, dims[l+1])
 * multiplier applied after the activation (training-mode Dropout(p=.5), layers.py:143-147). */
int dn_mini_mlp_fwd(const float* const* src_host, const int* src_width_host, int nsrc,
                    const float* const* weight_host, const float* const* bias_host,
                    const int* dims_host, int n_layers, const float* const* drop_mask_host,
                    const float* residual, int64_t V, float* const* hidden_out_host, float* out,
                    void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* Backward of dn_mini_mlp_fwd.  hidden[l] = h_{l+1} saved by the forward.  grad_src[s] written
 * (residual gradient is NOT added here); grad_weight / grad_bias ACCUMULATED. */
int dn_mini_mlp_bwd(const float* grad_out, const float* const* src_host, const int* src_width_host,
                    int nsrc, const float* const* weight_host, const int* dims_host, int n_layers,
                    const float* const* hidden_host, const float* const* drop_mask_host, int64_t V,
                    float* const* grad_src_host, float* const* grad_weight_host,
                    float* const* grad_bias_host, void* workspace, int64_t ws_bytes, int engine,
                    dn_stream_t stream);

/* layers.py:200-241 DiffusionNetBlock.forward for one mesh (eval mode: no dropout, nothing
 * saved).  L is unused by the spectral method and is not passed. */
int dn_block_fwd(const float* x_in, const float* mass, const float* evals, const float* evecs,
                 const dn_csr* grad, const dn_block_params* params, int64_t V, int K, int C,
                 float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* Profiling hook: the same launch sequence as dn_block_fwd with CUDA events recorded on `stream` between its stages;
 * SYNCHRONISES on the last event and writes DN_PROFILE_STAGES host floats (milliseconds):
 *   [0] to_basis (split-V partials)  [1] partial reduction + exp(-lambda t) scale when it is a separate launch
 *   (SIMT engine; 0 on the tensor-core path, where it is part of [2])  [2] weight split/pack (+ reduction and scale)
 *   [3] from_basis (+ [P|Q]) chain   [4] sparse gradient gather + inner product + tanh   [5] MiniMLP chain + skip
 * (bench.py reports each stage's roofline from these).  Not for use inside CUDA-graph capture. */
#define DN_PROFILE_STAGES 6
int dn_block_fwd_profile(const float* x_in, const float* mass, const float* evals, const float* evecs,
                         const dn_csr* grad, const dn_block_params* params, int64_t V, int K, int C,
                         float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream,
                         float* stage_ms_host);

/* Operator construction, the per-vertex part (SURVEY.md 8f-4): geometry.py:198-207 `edge_tangent_vectors` +
 * geometry.py:209-273 `build_grad` on the device, straight into dn_csr arrays.  `edges` is the reference's (2, E) int64
 * tensor (row 0 tails, row 1 tips, any order; self loops are skipped as in :228).  Pass either `edge_tangent` (E, 2)
 * as `build_grad` receives it, or NULL with `verts` (V, 3) and `frames` (V, 3, 3) to have it computed.  Row v of the
 * result holds the entry of v itself followed / surrounded by its neighbours, columns sorted; capacity E + V entries,
 * the actual count is rowptr_out[V] (device).  fp64 2x2 solves like numpy.  workspace: 4 * V bytes. */
int dn_build_grad(const float* verts, const float* frames, const float* edge_tangent, const int64_t* edges, int64_t E,
                  int64_t V, int32_t* rowptr_out, int32_t* colidx_out, float* vals_out, void* workspace,
                  int64_t ws_bytes, dn_stream_t stream);

/* ---- batches of independent meshes in one launch sequence (BASELINE config 4; SURVEY.md 8e) -------------------
 * The reference loops over the batch dimension with one set of operators per mesh (layers.py:217-222; a DataLoader
 * of batch_size None in every experiment).  Here a batch is ONE vertex range: mesh b occupies rows
 * [row_begin[b], row_begin[b] + n_rows[b]) of every (V, .) array; row_begin[b] is a multiple of 128 (a 128-row tile
 * never straddles two meshes); rows in the padding between meshes carry mass 0, basis 0 and no CSR entries; the CSR
 * is block diagonal with batch-global column indices; evals is (n_meshes, K).  Every per-vertex stage (gather,
 * MiniMLP) then runs as one launch over the whole range, and the per-mesh spectral stages run grouped:
 * to_basis CTAs never cross a mesh (tb_rows), the spectral multiplier is packed once per mesh and the from_basis chain
 * picks its weights per tile (tile_mesh).  Device arrays are built once per batch from dn_mesh_batch_plan's output. */
typedef struct dn_mesh_batch {
  int32_t n_meshes;
  int32_t n_tb_ctas;             /* CTAs of the grouped to_basis launch (<= 1024)                             */
  const int32_t* tile_mesh;      /* device [V / 128]: mesh of every 128-row tile                              */
  const int32_t* tb_rows;        /* device [2 * n_tb_ctas]: row range [begin, end) of each to_basis CTA       */
  const int32_t* mesh_cta_begin; /* device [n_meshes + 1]: the CTAs of mesh b are [begin[b], begin[b+1])      */
} dn_mesh_batch;

/* HOST-side planner (all pointers are HOST pointers): lays n_meshes meshes of n_rows_host[b] vertices out in one
 * row range (each start rounded up to 128) and splits them over about sm_count to_basis CTAs.
 * Outputs (caller-allocated): row_begin_host [n_meshes + 1] (last = padded total V), tile_mesh_host [V / 128],
 * tb_rows_host [2 * 1024], mesh_cta_begin_host [n_meshes + 1].  Returns the number of to_basis CTAs or DN_ERR_*. */
int dn_mesh_batch_plan(int n_meshes, const int32_t* n_rows_host, int sm_count, int32_t* row_begin_host,
                       int32_t* tile_mesh_host, int32_t* tb_rows_host, int32_t* mesh_cta_begin_host);

/* dn_block_fwd over a batch laid out as above (V = padded total, a multiple of 128).  Tensor-core engines only
 * (DN_ERR_UNSUPPORTED otherwise and for shapes outside the fused kernels' envelope: the caller loops over meshes). */
int dn_block_fwd_batched(const float* x_in, const float* mass, const float* evals, const float* evecs,
                         const dn_csr* grad, const dn_block_params* params, const dn_mesh_batch* batch, int64_t V,
                         int K, int C, float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

/* layers.py:44-67 LearnedTimeDiffusion over every mesh of a batch laid out as above, differentiable: the training
 * counterpart of the spectral stage of dn_block_fwd_batched.  evals is (n_meshes, K); time (C) is clamped in place
 * (layers.py:48-49).  x_spec_out (n_meshes, K, C) optional: mesh b's un-scaled spectral coefficients, saved for the
 * backward pass.  The launch count does not depend on the number of meshes.  Tensor-core engines only, and only shapes
 * whose from_basis chain picks its weights per tile: DN_ERR_UNSUPPORTED otherwise (the SIMT engine, K = 32, ...), with
 * nothing enqueued (the caller then loops over the meshes with dn_learned_time_diffusion_fwd). */
int dn_learned_time_diffusion_fwd_batched(const float* x, const float* mass, const float* evals, const float* evecs,
                                          float* time, const dn_mesh_batch* batch, int64_t V, int K, int C,
                                          float* x_diffuse, float* x_spec_out, void* workspace, int64_t ws_bytes,
                                          int engine, dn_stream_t stream);

/* Backward of the above w.r.t. x and time; x_spec is what the forward wrote to x_spec_out.  grad_x is written (exactly 0
 * on padding rows); grad_time (C) is ACCUMULATED into (+=), summed over the meshes in a fixed order (bit-reproducible).
 * Same support rules as the forward. */
int dn_learned_time_diffusion_bwd_batched(const float* grad_out, const float* mass, const float* evals,
                                          const float* evecs, const float* time, const float* x_spec,
                                          const dn_mesh_batch* batch, int64_t V, int K, int C, float* grad_x,
                                          float* grad_time, void* workspace, int64_t ws_bytes, int engine,
                                          dn_stream_t stream);

/* Linear head fused behind a block (SURVEY.md 8f-1): `DiffusionNet.last_lin` (layers.py:366-370 -- the nn.Linear applied
 * to the last block's output) computed in the epilogue of that block's MiniMLP chain, in exact fp32, so that the
 * C_width-wide block output is never written: out_head[v][o] = bias[o] + sum_c weight[o][c] * block_out[v][c]. */
typedef struct dn_head {
  const float* weight;  /* (n_out, C) nn.Linear layout */
  const float* bias;    /* (n_out) or NULL             */
  int32_t n_out;        /* 1..8                        */
  float* out;           /* (V, n_out), row stride ld_out floats */
  int64_t ld_out;
} dn_head;

/* dn_block_fwd / dn_block_fwd_batched with options: `batch` may be NULL (one mesh), `head` may be NULL.  With a head, `out`
 * (the block output) may be NULL; DN_ERR_UNSUPPORTED when the MiniMLP does not run on the fused tensor-core chain (the
 * caller then applies the head as a separate layer). */
int dn_block_fwd_ex(const float* x_in, const float* mass, const float* evals, const float* evecs, const dn_csr* grad,
                    const dn_block_params* params, const dn_mesh_batch* batch, const dn_head* head, int64_t V, int K,
                    int C, float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFUSION_NET_B200_H */
