// Internal (non-ABI) declarations shared by the SIMT kernels, the tcgen05 kernels and the
// C-ABI glue.  Everything here is device-pointer based; no torch types anywhere in csrc/.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "../../include/diffusion_net_b200.h"

#define DN_MAX_SRC 3
#define DN_MAX_LAYERS 8

#define DN_CUDA_TRY(expr)                          \
  do {                                             \
    cudaError_t _e = (expr);                       \
    if (_e != cudaSuccess) return (int)_e;         \
  } while (0)

extern long long g_dn_launches;   // kernels launched by this library (reported by bench.py)

#define DN_LAUNCH_CHECK()                          \
  do {                                             \
    cudaError_t _e = cudaGetLastError();           \
    if (_e != cudaSuccess) return (int)_e;         \
    ++g_dn_launches;                               \
  } while (0)

// One affine layer applied to 128-row tiles of vertices:  out = epi(A @ W^T + bias)
//   A = concat_s src[s] (layer 0) -- or the previous layer's output inside a fused chain.
struct DnLayer {
  const float* W;        // nn.Linear layout [N][K] (ldw = K) when !w_trans; [K][N] (ldw = N) when w_trans
  int64_t ldw;
  int w_trans;
  const float* W2;       // optional second block: !w_trans: output rows n >= n_split come from W2[n - n_split]
  int n_split;           //   (stacks [A_re; A_im] without a copy);  w_trans: input rows k >= n_split come from W2[k - n_split]
  const float* prepacked;  // optional: weights already in the tensor-core layout (tc_pack_layers)
  int pack_fmt;            // layout of `prepacked`: 0 = 16-wide chunks of [tf32 hi | tf32 lo] (round-1 kernels, 3xTF32);
                           //   1 = 32-wide stages of [tf32 hi | bf16 (hi ; lo)] (rows_chain3_kernel, TF32 + bf16 corrections);
                           //   2 = 64-wide stages of bf16 (rows_chain16_kernel, DN_ENGINE_BF16)
  const float* bias;     // [N] or null
  int relu;
  const float* emul;     // optional elementwise multiplier [V][N] applied after the activation
  const float* relu_mask_src;  // optional [V][N]: multiply by (src > 0)   (backward of ReLU)
  const float* row_scale;      // optional [V]: multiply rows (mass, backward of to_basis)
  const float* residual; // optional [V][N] added last (times res_scale)
  int64_t ld_res;
  float res_scale;
  float* out;            // optional [V][N] (ld_out); null => stays on chip (fused chain only)
  int64_t ld_out;
  int K, N;
  // mesh batches (layer 0 of a chain only): `prepacked` holds one packed matrix per mesh, group_stride floats apart,
  // and 128-row tile t uses matrix tile_group[t] (device array)
  const int32_t* tile_group;
  int64_t group_stride;
  // complex inner-product epilogue (last layer of a chain only; layers.py:128-130).  The layer computes
  // [Bre | Bim] = in @ W^T with N/2 columns each for N/2 channels; the output (N/2 wide) is
  //   tanh(gX * Bre + gY * Bim),  gX = dots_src[:, c], gY = dots_src[:, dots_gy_col + c]   (row stride ld_dots)
  const float* dots_src;
  int64_t ld_dots;
  int dots_gy_col;
  // weights given as the pair (W = A_re, W2 = A_im) of SpatialGradientFeatures acting on [gX | gY]: see PackJob::rot_C
  int rot_C, rot_ch0;
  // linear head fused behind the last layer's epilogue (DiffusionNet.last_lin, layers.py:366-370): after bias / residual the
  // N-wide row y is NOT stored (out may be null); head_out[v][o] = head_b[o] + sum_n head_w[o][n] * y[n], o < head_n <= 8,
  // exact fp32 FMAs in the output warps
  const float* head_w;
  const float* head_b;
  float* head_out;
  int64_t ld_head_out;
  int head_n;
};

#ifdef __CUDACC__
// tanh of the gradient features (layers.py:130): 1 - 2 / (exp(2x) + 1) with the fast exp / divide; absolute error
// <= ~1.5e-7 over the whole range, saturates to +-1, NaN propagates.  Every kernel that forms features uses this one.
__device__ __forceinline__ float dn_feat_tanh(float x) {
  const float e = __expf(2.f * x);
  return 1.f - __fdividef(2.f, e + 1.f);
}
#endif

struct DnRowsSrc {
  const float* ptr[DN_MAX_SRC];
  int width[DN_MAX_SRC];
  int64_t ld[DN_MAX_SRC];
  int nsrc;
};

// ---- SIMT engine (dn_simt.cu) ----
int simt_rows_gemm(const DnRowsSrc& src, const DnLayer& layer, int64_t V, cudaStream_t st);
// out[i][j] (ld_out) (+)= sum_v A[v][i] * scale[v] * B[v][j];  partial sums staged in ws.
int simt_atb(const float* A, int64_t lda, int I, const float* B, int64_t ldb, int J, const float* scale,
             int64_t V, float* out, int64_t ld_out, int accumulate, float* ws, int64_t ws_floats,
             cudaStream_t st);
int simt_atb_partial_st(const float* A, int64_t lda, int I, const float* B, int64_t ldb, int J, const float* scale,
                        int64_t V, float* ws, int64_t ws_floats, int* P_out, cudaStream_t st);
int simt_colsum(const float* A, int64_t lda, int N, int64_t V, float* out, int accumulate, cudaStream_t st);

// ---- shared small kernels (dn_simt.cu) ----
// S[k][c] = exp(-evals[k]*max(t[c],1e-8)) * sum_p partial[p][k][c]; optionally writes the raw sum
// (x_spec) and the clamped time back.  s_trans: write S as [c][k].
int launch_spectral_scale(const float* partial, int P, const float* evals, float* time, int K, int C,
                          float* x_spec_out, float* S_out, int clamp_writeback, cudaStream_t st);
int launch_reduce_partials(const float* partial, int P, int64_t n, float* out, cudaStream_t st);
int launch_reduce_partials_ld(const float* partial, int P, int rows, int cols, float* out, int64_t ld_out,
                              int accumulate, cudaStream_t st);
int launch_csr_from_coo(const int64_t* rows, const int64_t* cols, const float* vx, const float* vy,
                        int64_t nnz, int64_t V, int32_t* rowptr, int32_t* colidx, float* vals, cudaStream_t st);
int launch_compute_hks(const float* evals, const float* evecs, const float* scales, int64_t V, int K, int S,
                       float* out, cudaStream_t st);
int launch_build_grad(const float* verts, const float* frames, const float* edge_tangent, const int64_t* edges, int64_t E,
                      int64_t V, int32_t* rowptr, int32_t* colidx, float* vals, int32_t* cursor, cudaStream_t st);
int launch_csr_transpose(const dn_csr* in, int64_t V, int32_t* rowptr_t, int32_t* colidx_t, float* vals_t,
                         int32_t* cursor, cudaStream_t st);
int launch_grad_spmm_pair(const dn_csr* g, const float* x, int64_t V, int C, float* out_vc2, cudaStream_t st);
// R-order fused features: feat = tanh(gX*Bre + gY*Bim) from gathers of xd, P, Q (pq = [P|Q], ld 2C or C).
int launch_spmm_features(const dn_csr* g, const float* xd, const float* pq, int rotations, int64_t V, int C,
                         float* feat, cudaStream_t st);
// gxy[v] = [ (gradX @ x)[v] | (gradY @ x)[v] ]  (V x 2C, row-major): the gather of the tensor-core gradient-features
// route (C = 128 or 256)
int launch_spmm_gxy(const dn_csr* g, const float* x, int64_t V, int C, float* gxy, cudaStream_t st);
int launch_features_bwd_local(const dn_csr* g, const float* xd, const float* pq, const float* feat,
                              const float* dfeat, int rotations, int64_t V, int C, float* U /*V x 4C*/,
                              cudaStream_t st);
int launch_features_bwd_transpose(const dn_csr* gt, const float* U, int rotations, int64_t V, int C,
                                  float* dxd /*V x C*/, float* dP, float* dQ /*V x C each, leading dim ld_pq*/,
                                  int64_t ld_pq, cudaStream_t st);
int launch_deinterleave_vc2(const float* vc2, int64_t V, int C, float* g01 /*V x 2C*/, cudaStream_t st);
int launch_complex_dots_tanh(const float* g01, const float* b01, int64_t V, int C, float* out, cudaStream_t st);
int launch_spectral_bwd(const float* gs_partial, int P, const float* evals, const float* time,
                        const float* x_spec, int K, int C, float* dS /*K x C*/, float* grad_time /*+=*/,
                        cudaStream_t st);

// ---- tcgen05 engine (dn_tc.cu) ----
bool tc_supported_device();
// Fused chain of up to DN_MAX_LAYERS layers over 128-row tiles; layer 0 reads `src`.
int tc_rows_chain(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int64_t V, int passes /*3 or 1*/,
                  void* ws, int64_t ws_bytes, cudaStream_t st);
// `passes`: 3 = 3xTF32-grade (fp32 parity), 1 = single-pass TF32, DN_PASSES_BF16 = single-pass bf16 (DN_ENGINE_BF16)
#define DN_PASSES_BF16 16
int tc_rows_chain_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int passes = 3);
// packed-weight layout the kernel that will run this chain expects (sets layers[i].pack_fmt; call before tc_pack_layers)
void tc_choose_pack_fmt(const DnRowsSrc& src, DnLayer* layers, int n_layers, int passes = 3);
// partial[p][k][c] for p < *P_out
// `values` may be a column slice (row stride ld_values >= C) and a partial a slice of a wider one (row stride ldp):
// C_width = 256 runs as two 128-column launches into the same [P][K][256] partials.  0 = contiguous (== C).
int tc_to_basis_partial(const float* values, const float* basis, const float* massvec, int64_t V, int K, int C,
                        float* partial, int* P_out, int passes, cudaStream_t st, int64_t ld_values = 0, int64_t ldp = 0,
                        const int32_t* cta_rows = nullptr, int n_ctas = 0);
int tc_to_basis_supported(int K, int C);
int64_t tc_chain_ws_bytes(const DnLayer* layers, int n_layers);
// mesh batches: pack S_b = exp(-evals_b t) * (partials of mesh b) for every mesh as layer0's per-mesh weights
// (ws: n_meshes * tc_chain_ws_bytes(layer0, 1) bytes); sets layer0->prepacked / tile_group / group_stride.
// x_spec_out (optional, [n_meshes][K][N]) receives every mesh's reduced, unscaled coefficients.
int tc_pack_spectral_batched(DnLayer* layer0, int n_meshes, void* ws, int64_t ws_bytes, const float* partial,
                             const int32_t* mesh_cta_begin, const float* evals, float* time, int clamp_writeback,
                             const int32_t* tile_mesh, cudaStream_t st, float* x_spec_out = nullptr);
// mesh batches, backward (two launches): from the partials of Phi_b^T g_b, pack dS_b = exp(-evals_b t) * Gs_b as layer0's
// per-mesh weights (as above) and add sum_b sum_k Gs_b * (-lambda_bk) * E_b * x_spec_b to grad_time in a fixed order.
// dt_scratch: tc_spectral_bwd_batched_scratch_floats(n_meshes, K, N) floats.
#define DN_SPEC_BWD_KROWS 4
int64_t tc_spectral_bwd_batched_scratch_floats(int n_meshes, int K, int N);
int tc_spectral_bwd_batched(DnLayer* layer0, int n_meshes, void* ws, int64_t ws_bytes, const float* partial,
                            const int32_t* mesh_cta_begin, const float* evals, const float* time, const float* x_spec,
                            float* dt_scratch, float* grad_time, const int32_t* tile_mesh, cudaStream_t st);
// the chain kernels that can pick layer-0 weights per tile (tile_group): chain3, and chain16 on the bf16 engine
int tc_grouped_chain_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int passes);
// one launch: pack the weights of n layers into ws and set layers[i].prepacked
int tc_pack_layers(DnLayer* layers, int n_layers, void* ws, int64_t ws_bytes, cudaStream_t st);
// same, with layers[0] (w_trans, K = eigen count, N = channels) replaced by the spectral multiplier
//   S[k][n] = exp(-evals[k] * max(time[n], 1e-8)) * sum_p partial[p][k][n]    (one launch for scale + pack)
int tc_pack_layers_spectral(DnLayer* layers, int n_layers, void* ws, int64_t ws_bytes, const float* partial, int P,
                            const float* evals, float* time, int clamp_writeback, cudaStream_t st);
