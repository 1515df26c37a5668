// C-ABI entry points (include/diffusion_net_b200.h).  Argument checking, workspace carving and
// the kernel sequence of each reference function; no torch types, no hidden synchronisation.
#include "dn_internal.h"
#include <stdio.h>
#include <stdlib.h>
#include <vector>
#include <string.h>

namespace {

struct Bump {
  char* base;
  int64_t size, off;
  Bump(void* p, int64_t n) : base(static_cast<char*>(p)), size(n), off(0) {}
  float* take(int64_t floats) {
    const int64_t bytes = (floats * 4 + 255) / 256 * 256;
    if (!base || off + bytes > size) return nullptr;
    float* r = reinterpret_cast<float*>(base + off);
    off += bytes;
    return r;
  }
  int64_t left_floats() const { return (size - off) / 4; }
};

constexpr int64_t kPartialFloats = 16ll << 20;  // 64 MiB split-V partial sums

// The engine as the helpers below take it, resolved once per entry point before anything is enqueued: 0 runs the exact
// fp32 SIMT kernels, otherwise the tensor-core pass count (3, 1 or DN_PASSES_BF16).  A tensor-core engine on a device
// without tcgen05 is DN_ERR_NOT_SM100: there is no multi-backend dispatch.
int resolve_engine(int engine, int* tc) {
  *tc = engine == DN_ENGINE_TC3X ? 3 : engine == DN_ENGINE_TC1X ? 1 : engine == DN_ENGINE_BF16 ? DN_PASSES_BF16 : 0;
  return (*tc && !tc_supported_device()) ? DN_ERR_NOT_SM100 : DN_OK;
}

// A tensor-core engine was requested but this contraction is outside the tcgen05 kernels' envelope and runs the exact
// fp32 SIMT kernel instead (same result class or better, slower).  Said once per shape on stderr; DN_STRICT_TC=1 turns
// it into DN_ERR_UNSUPPORTED so that a deployment never runs the slow path unnoticed.
int note_simt_fallback(const char* what, int K, int N) {
  static int strict = -1;
  if (strict < 0) { const char* e = getenv("DN_STRICT_TC"); strict = (e && atoi(e)) ? 1 : 0; }
  static int seen[64][2];
  static int nseen = 0;
  bool first = true;
  for (int i = 0; i < nseen; ++i) if (seen[i][0] == K && seen[i][1] == N) first = false;
  if (first && nseen < 64) {
    seen[nseen][0] = K; seen[nseen][1] = N; ++nseen;
    fprintf(stderr, "diffusion_net_b200: %s with K=%d, N=%d is outside the tensor-core kernels' envelope; running the exact "
                    "fp32 SIMT kernel%s\n", what, K, N, strict ? " is refused (DN_STRICT_TC=1)" : "");
  }
  return strict ? DN_ERR_UNSUPPORTED : DN_OK;
}

inline DnLayer make_layer(const float* W, int64_t ldw, int w_trans, const float* bias, int relu, int K, int N,
                          float* out, int64_t ld_out) {
  DnLayer L;
  memset(&L, 0, sizeof(L));
  L.W = W; L.ldw = ldw; L.w_trans = w_trans; L.bias = bias; L.relu = relu; L.K = K; L.N = N;
  L.out = out; L.ld_out = ld_out; L.res_scale = 1.f;
  return L;
}

inline DnRowsSrc one_src(const float* p, int width, int64_t ld) {
  DnRowsSrc s;
  memset(&s, 0, sizeof(s));
  s.ptr[0] = p; s.width[0] = width; s.ld[0] = ld; s.nsrc = 1;
  return s;
}

// run a chain of layers; tensor-core engine `tc` (resolve_engine) when it supports the shapes, exact SIMT otherwise.
// `tmp0/tmp1` are V x maxN ping-pong buffers used only by the unfused SIMT route.
int run_chain(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int64_t V, int tc, float* tmp0, float* tmp1,
              void* tc_ws, int64_t tc_ws_bytes, cudaStream_t st) {
  if (tc && tc_rows_chain_supported(src, layers, n_layers, tc) == DN_OK)
    return tc_rows_chain(src, layers, n_layers, V, tc, tc_ws, tc_ws_bytes, st);
  // not fusable as a whole (e.g. a 256-wide layer inside a chain): layer by layer, each on the
  // tensor-core kernel when its shape allows, on the exact SIMT kernel otherwise
  DnRowsSrc cur = src;
  for (int l = 0; l < n_layers; ++l) {
    DnLayer L = layers[l];
    float* o = L.out;
    int64_t ldo = L.ld_out;
    if (!o) {
      o = (l & 1) ? tmp1 : tmp0;
      ldo = L.N;
      if (!o) return DN_ERR_WORKSPACE;
    }
    L.out = o; L.ld_out = ldo;
    int rc;
    if (tc && tc_rows_chain_supported(cur, &L, 1, tc) == DN_OK)
      rc = tc_rows_chain(cur, &L, 1, V, tc, tc_ws, tc_ws_bytes, st);
    else {
      if (tc && (rc = note_simt_fallback("a dense layer", L.K, L.N))) return rc;
      rc = simt_rows_gemm(cur, L, V, st);
    }
    if (rc) return rc;
    cur = one_src(o, L.N, ldo);
  }
  return DN_OK;
}

// shapes the split-V tensor-core to_basis takes: up to 128 columns in one launch, wider (C_width = 256) in 128-column
// slices
bool to_basis_tc_fits(int K, int C) {
  return tc_to_basis_supported(K, C) == DN_OK || (C > 128 && C % 128 == 0 && tc_to_basis_supported(K, 128) == DN_OK);
}

// split-V to_basis partials on the tensor cores, for a shape to_basis_tc_fits accepts: wider than one accumulator set,
// each 128-column slice is its own launch into the shared [P][K][C] partials.  With `batch`, grouped over a mesh batch:
// every CTA reduces a row range inside one mesh (batch->tb_rows) into its own K x C partial.
int to_basis_tc(const float* values, const float* basis, const float* massvec, int64_t V, int K, int C, float* partial,
                int* P, int tc, cudaStream_t st, const dn_mesh_batch* batch = nullptr) {
  const int32_t* cta_rows = batch ? batch->tb_rows : nullptr;
  const int n_ctas = batch ? batch->n_tb_ctas : 0;
  if (tc_to_basis_supported(K, C) == DN_OK)
    return tc_to_basis_partial(values, basis, massvec, V, K, C, partial, P, tc, st, 0, 0, cta_rows, n_ctas);
  for (int c0 = 0; c0 < C; c0 += 128) {
    const int rc = tc_to_basis_partial(values + c0, basis, massvec, V, K, 128, partial + c0, P, tc, st, C, C, cta_rows,
                                       n_ctas);
    if (rc) return rc;
  }
  return DN_OK;
}

int to_basis_partials(const float* values, const float* basis, const float* massvec, int64_t V, int K, int C,
                      float* partial, int64_t partial_floats, int* P, int tc, cudaStream_t st) {
  if (tc && to_basis_tc_fits(K, C) && (int64_t)148 * K * C <= partial_floats)
    return to_basis_tc(values, basis, massvec, V, K, C, partial, P, tc, st);
  if (tc) { const int rc = note_simt_fallback("to_basis", K, C); if (rc) return rc; }
  // out[k][c] = sum_v basis[v][k] * (mass[v] * values[v][c])
  return simt_atb_partial_st(basis, K, K, values, C, C, massvec, V, partial, partial_floats, P, st);
}

// out[i][j] (ld_out) (+)= sum_v A[v][i] * B[v][j]   (weight gradients: A = dz, B = layer input).
// Tensor cores (the split-V to_basis kernel, reference geometry.py:572-583 has the same contraction) when both
// operands are contiguous and at most 128 wide; the exact SIMT kernel otherwise.
int atb(const float* A, int64_t lda, int I, const float* B, int64_t ldb, int J, int64_t V, float* out, int64_t ld_out,
        int accumulate, float* part, int64_t part_floats, int tc, cudaStream_t st) {
  if (tc && lda == I && ldb == J && tc_to_basis_supported(I, J) == DN_OK && (int64_t)148 * I * J <= part_floats) {
    int P = 0;
    int rc = tc_to_basis_partial(B, A, nullptr, V, I, J, part, &P, tc, st);
    if (rc == DN_OK) return launch_reduce_partials_ld(part, P, I, J, out, ld_out, accumulate, st);
    if (rc != DN_ERR_UNSUPPORTED) return rc;
  }
  if (tc) { const int rc = note_simt_fallback("a weight gradient", I, J); if (rc) return rc; }
  return simt_atb(A, lda, I, B, ldb, J, nullptr, V, out, ld_out, accumulate, part, part_floats, st);
}

// A mesh batch (dn_mesh_batch_plan) laid out as one vertex range, and the grouped to_basis of `values` over it, checked
// before anything is enqueued: every descriptor field set, whole 128-row tiles, 16-byte aligned `values` / `evecs`,
// K and C inside the split-V kernel.
int check_batch(const dn_mesh_batch* batch, const float* values, const float* evecs, int64_t V, int K, int C) {
  if (!batch || batch->n_meshes < 1 || batch->n_tb_ctas < 1 || !batch->tile_mesh || !batch->tb_rows ||
      !batch->mesh_cta_begin)
    return DN_ERR_INVALID_ARGUMENT;
  if ((V % 128) || V >= (1ll << 31) - 256 || (C % 4) || (reinterpret_cast<uintptr_t>(values) & 15) ||
      (reinterpret_cast<uintptr_t>(evecs) & 15) || !to_basis_tc_fits(K, C))
    return DN_ERR_UNSUPPORTED;
  return DN_OK;
}

// Support checks of the grouped spectral stage (learned-time diffusion over a mesh batch), all made before anything is
// enqueued: the batch, and a from_basis chain `L` that picks its weights per tile.  Chooses L's pack format.
int grouped_spectral_check(const float* values, const float* evecs, const dn_mesh_batch* batch, int64_t V, int K, int C,
                           int tc, DnLayer* L) {
  const int rc = check_batch(batch, values, evecs, V, K, C);
  if (rc) return rc;
  const DnRowsSrc src = one_src(evecs, K, K);
  if (!tc || tc_grouped_chain_supported(src, L, 1, tc) != DN_OK) return DN_ERR_UNSUPPORTED;
  tc_choose_pack_fmt(src, L, 1, tc);
  return DN_OK;
}

}  // namespace

long long g_dn_launches = 0;
// bring-up: device time of the x-only gather inside stage [4] of the last dn_block_fwd_profile call (tools only)
static cudaEvent_t g_gf_ev = nullptr;
static float g_gf_gather_ms = 0.f;
static bool g_gf_recorded = false;
extern "C" float dn_debug_gf_gather_ms(void) { return g_gf_gather_ms; }

extern "C" {

int dn_abi_version(void) { return DN_ABI_VERSION; }

int64_t dn_kernel_launch_count(void) { return (int64_t)g_dn_launches; }

const char* dn_error_string(int code) {
  switch (code) {
    case DN_OK: return "ok";
    case DN_ERR_INVALID_ARGUMENT: return "diffusion_net_b200: invalid argument";
    case DN_ERR_UNSUPPORTED: return "diffusion_net_b200: unsupported shape/engine";
    case DN_ERR_WORKSPACE: return "diffusion_net_b200: workspace too small (see dn_workspace_bytes)";
    case DN_ERR_NOT_SM100: return "diffusion_net_b200: tensor-core engine needs an sm_100 GPU";
    default: break;
  }
  if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
  return "diffusion_net_b200: unknown error";
}

int dn_device_query(int device, int* sm_count, int* cc, int64_t* smem_optin_bytes) {
  cudaDeviceProp p;
  DN_CUDA_TRY(cudaGetDeviceProperties(&p, device));
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (cc) *cc = p.major * 10 + p.minor;
  if (smem_optin_bytes) *smem_optin_bytes = (int64_t)p.sharedMemPerBlockOptin;
  return DN_OK;
}

int64_t dn_workspace_bytes(int64_t V, int K, int C) {
  if (V < 0 || K < 0 || C <= 0) return -1;
  const int64_t vc = ((V + 127) / 128 * 128) * (int64_t)C * 4;
  return kPartialFloats * 4 + 14 * (vc + 256) + (8ll << 20) + (int64_t)K * C * 16;
}

int dn_csr_from_coo(const int64_t* rows, const int64_t* cols, const float* vx, const float* vy, int64_t nnz,
                    int64_t V, int32_t* rowptr, int32_t* colidx, float* vals, dn_stream_t stream) {
  if (nnz < 0 || V < 0 || !rowptr || (nnz > 0 && (!rows || !cols || !vx || !colidx || !vals)))
    return DN_ERR_INVALID_ARGUMENT;
  if (nnz >= (1ll << 31) || V >= (1ll << 31)) return DN_ERR_UNSUPPORTED;
  return launch_csr_from_coo(rows, cols, vx, vy, nnz, V, rowptr, colidx, vals, (cudaStream_t)stream);
}

int64_t dn_patch_build(int64_t V, const int32_t* rowptr, const int32_t* colidx, int max_targets, int max_src,
                       int32_t* tgt_ptr, int32_t* tgt, int32_t* src_ptr, int32_t* src_rows, int32_t* ent_ptr,
                       uint8_t* lcol, int32_t* perm, int32_t* max_src_out) {
  if (V < 0 || !rowptr || max_targets < 1 || max_src < 1 || max_src > 256 || !tgt_ptr || !tgt || !src_ptr ||
      !ent_ptr || !max_src_out || (V > 0 && rowptr[V] > 0 && (!colidx || !src_rows || !lcol || !perm)))
    return DN_ERR_INVALID_ARGUMENT;
  if (V >= (1ll << 31) - 1) return DN_ERR_UNSUPPORTED;
  // state: 0 free, 1 queued by the patch being grown, 2 assigned
  std::vector<int32_t> stamp((size_t)V, -1), lidx((size_t)V, 0), seeds, q;
  std::vector<uint8_t> state((size_t)V, 0);
  size_t seed_head = 0;
  int64_t scan = 0, np = 0, nt = 0, nsr = 0, ne = 0;
  int32_t worst = 0;
  tgt_ptr[0] = 0; src_ptr[0] = 0; ent_ptr[0] = 0;
  while (nt < V) {
    int32_t s = -1;
    while (seed_head < seeds.size()) {                       // prefer a vertex next to an earlier patch
      const int32_t c = seeds[seed_head++];
      if (state[c] == 0) { s = c; break; }
    }
    if (s < 0) {
      while (state[scan] != 0) ++scan;
      s = (int32_t)scan;
    }
    q.clear();
    q.push_back(s);
    state[s] = 1;
    size_t qh = 0;
    int nsrc = 0, ntg = 0;
    while (qh < q.size() && ntg < max_targets) {
      const int32_t v = q[qh++];
      const int32_t rs = rowptr[v], re = rowptr[v + 1];
      if (re - rs > max_src) return DN_ERR_UNSUPPORTED;
      int newc = 0;
      for (int32_t e = rs; e < re; ++e) newc += (stamp[colidx[e]] != (int32_t)np);
      if (nsrc + newc > max_src) {                           // does not fit here: a later patch takes it
        state[v] = 0;
        seeds.push_back(v);
        continue;
      }
      state[v] = 2;
      tgt[nt++] = v;
      ++ntg;
      for (int32_t e = rs; e < re; ++e) {
        const int32_t c = colidx[e];
        if (stamp[c] != (int32_t)np) {
          stamp[c] = (int32_t)np;
          lidx[c] = nsrc++;
          src_rows[nsr++] = c;
        }
        lcol[ne] = (uint8_t)lidx[c];
        perm[ne] = e;
        ++ne;
      }
      ent_ptr[nt] = (int32_t)ne;
      for (int32_t e = rs; e < re; ++e) {
        const int32_t c = colidx[e];
        if (c < V && state[c] == 0) { state[c] = 1; q.push_back(c); }
      }
    }
    for (; qh < q.size(); ++qh) {                            // frontier we did not get to: seeds of the next patches
      const int32_t v = q[qh];
      if (state[v] == 1) { state[v] = 0; seeds.push_back(v); }
    }
    if (nsrc > worst) worst = nsrc;
    ++np;
    tgt_ptr[np] = (int32_t)nt;
    src_ptr[np] = (int32_t)nsr;
  }
  *max_src_out = worst;
  return np;
}

int dn_csr_transpose(const dn_csr* in, int64_t V, int32_t* rowptr_out, int32_t* colidx_out, float* vals_out,
                     void* workspace, int64_t ws_bytes, dn_stream_t stream) {
  if (!in || V < 0 || in->nnz < 0 || !rowptr_out || (in->nnz > 0 && (!in->rowptr || !in->colidx || !in->vals ||
                                                                        !colidx_out || !vals_out)))
    return DN_ERR_INVALID_ARGUMENT;
  if (in->nnz >= (1ll << 31) || V >= (1ll << 31) - 1) return DN_ERR_UNSUPPORTED;
  if (in->nnz > 0 && (!workspace || ws_bytes < (int64_t)sizeof(int32_t) * V)) return DN_ERR_WORKSPACE;
  return launch_csr_transpose(in, V, rowptr_out, colidx_out, vals_out, (int32_t*)workspace, (cudaStream_t)stream);
}

int dn_build_grad(const float* verts, const float* frames, const float* edge_tangent, const int64_t* edges, int64_t E,
                  int64_t V, int32_t* rowptr_out, int32_t* colidx_out, float* vals_out, void* workspace, int64_t ws_bytes,
                  dn_stream_t stream) {
  if (V < 0 || E < 0 || !rowptr_out || (V > 0 && (!colidx_out || !vals_out)) || (E > 0 && !edges) ||
      (E > 0 && !edge_tangent && (!verts || !frames)))
    return DN_ERR_INVALID_ARGUMENT;
  if (E + V >= (1ll << 31) || V >= (1ll << 31) - 1) return DN_ERR_UNSUPPORTED;
  if (V > 0 && (!workspace || ws_bytes < (int64_t)sizeof(int32_t) * V)) return DN_ERR_WORKSPACE;
  return launch_build_grad(verts, frames, edge_tangent, edges, E, V, rowptr_out, colidx_out, vals_out, (int32_t*)workspace,
                           (cudaStream_t)stream);
}

int dn_compute_hks(const float* evals, const float* evecs, const float* scales, int64_t V, int K, int S, float* out,
                   dn_stream_t stream) {
  if (V < 0 || K <= 0 || S < 0 || ((V > 0 && S > 0) && (!evals || !evecs || !scales || !out)))
    return DN_ERR_INVALID_ARGUMENT;
  return launch_compute_hks(evals, evecs, scales, V, K, S, out, (cudaStream_t)stream);
}

int dn_to_basis(const float* values, const float* basis, const float* massvec, int64_t V, int K, int C, float* out,
                void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!values || !basis || !out || V < 0 || K <= 0 || C <= 0) return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int64_t pf = ws.left_floats() < kPartialFloats ? ws.left_floats() : kPartialFloats;
  float* partial = ws.take(pf);
  if (!partial) return DN_ERR_WORKSPACE;
  int P = 0;
  if ((rc = to_basis_partials(values, basis, massvec, V, K, C, partial, pf, &P, tc, st))) return rc;
  return launch_reduce_partials(partial, P, (int64_t)K * C, out, st);
}

int dn_from_basis(const float* values, const float* basis, const float* row_scale, int64_t V, int K, int C,
                  float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!values || !basis || !out || V < 0 || K <= 0 || C <= 0) return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  DnRowsSrc src = one_src(basis, K, K);
  DnLayer L = make_layer(values, C, /*w_trans=*/1, nullptr, 0, K, C, out, C);
  L.row_scale = row_scale;
  return run_chain(src, &L, 1, V, tc, nullptr, nullptr, workspace, ws_bytes, (cudaStream_t)stream);
}

int dn_learned_time_diffusion_fwd(const float* x, const float* mass, const float* evals, const float* evecs,
                                  float* time, int64_t V, int K, int C, float* x_diffuse, float* x_spec_out,
                                  void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!x || !mass || !evals || !evecs || !time || !x_diffuse || V < 0 || K <= 0 || C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  float* S = ws.take((int64_t)K * C);
  const int64_t pf = ws.left_floats() / 2 < kPartialFloats ? ws.left_floats() / 2 : kPartialFloats;
  float* partial = ws.take(pf);
  if (!S || !partial) return DN_ERR_WORKSPACE;
  int P = 0;
  if ((rc = to_basis_partials(x, evecs, mass, V, K, C, partial, pf, &P, tc, st))) return rc;
  rc = launch_spectral_scale(partial, P, evals, time, K, C, x_spec_out, S, /*clamp_writeback=*/1, st);
  if (rc) return rc;
  DnRowsSrc src = one_src(evecs, K, K);
  DnLayer L = make_layer(S, C, 1, nullptr, 0, K, C, x_diffuse, C);
  return run_chain(src, &L, 1, V, tc, nullptr, nullptr, ws.base + ws.off, ws.size - ws.off, st);
}

int dn_learned_time_diffusion_bwd(const float* grad_out, const float* mass, const float* evals, const float* evecs,
                                  const float* time, const float* x_spec, int64_t V, int K, int C, float* grad_x,
                                  float* grad_time, void* workspace, int64_t ws_bytes, int engine,
                                  dn_stream_t stream) {
  if (!grad_out || !mass || !evals || !evecs || !time || !x_spec || !grad_x || !grad_time)
    return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  float* dS = ws.take((int64_t)K * C);
  const int64_t pf = ws.left_floats() / 2 < kPartialFloats ? ws.left_floats() / 2 : kPartialFloats;
  float* partial = ws.take(pf);
  if (!dS || !partial) return DN_ERR_WORKSPACE;
  int P = 0;
  if ((rc = to_basis_partials(grad_out, evecs, nullptr, V, K, C, partial, pf, &P, tc, st))) return rc;
  if (P > 4) {
    // spectral_bwd walks the partials serially per channel: with the 148 split-V partials of the tensor-core kernel that
    // took 4.5 ms (V = 7k); sum them first (coalesced, parallel) and hand it one
    float* red = ws.take((int64_t)K * C);
    if (!red) return DN_ERR_WORKSPACE;
    if ((rc = launch_reduce_partials(partial, P, (int64_t)K * C, red, st))) return rc;
    rc = launch_spectral_bwd(red, 1, evals, time, x_spec, K, C, dS, grad_time, st);
  } else {
    rc = launch_spectral_bwd(partial, P, evals, time, x_spec, K, C, dS, grad_time, st);
  }
  if (rc) return rc;
  DnRowsSrc src = one_src(evecs, K, K);
  DnLayer L = make_layer(dS, C, 1, nullptr, 0, K, C, grad_x, C);
  L.row_scale = mass;
  return run_chain(src, &L, 1, V, tc, nullptr, nullptr, ws.base + ws.off, ws.size - ws.off, st);
}

int dn_learned_time_diffusion_fwd_batched(const float* x, const float* mass, const float* evals, const float* evecs,
                                          float* time, const dn_mesh_batch* batch, int64_t V, int K, int C,
                                          float* x_diffuse, float* x_spec_out, void* workspace, int64_t ws_bytes,
                                          int engine, dn_stream_t stream) {
  if (!x || !mass || !evals || !evecs || !time || !x_diffuse || V < 0 || K <= 0 || C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  DnLayer L = make_layer(nullptr, C, /*w_trans=*/1, nullptr, 0, K, C, x_diffuse, C);
  int tc, rc = resolve_engine(engine, &tc);
  if (rc || (rc = grouped_spectral_check(x, evecs, batch, V, K, C, tc, &L))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int64_t pb = tc_chain_ws_bytes(&L, 1) * batch->n_meshes;
  float* pk = ws.take(pb / 4);
  float* partial = ws.take((int64_t)batch->n_tb_ctas * K * C);
  if (!pk || !partial) return DN_ERR_WORKSPACE;
  // (nothing has been enqueued up to here)
  int P = 0;
  if ((rc = to_basis_tc(x, evecs, mass, V, K, C, partial, &P, tc, st, batch))) return rc;
  if ((rc = tc_pack_spectral_batched(&L, batch->n_meshes, pk, pb, partial, batch->mesh_cta_begin, evals, time,
                                     /*clamp_writeback=*/1, batch->tile_mesh, st, x_spec_out)))
    return rc;
  return tc_rows_chain(one_src(evecs, K, K), &L, 1, V, tc, ws.base + ws.off, ws.size - ws.off, st);
}

int dn_learned_time_diffusion_bwd_batched(const float* grad_out, const float* mass, const float* evals,
                                          const float* evecs, const float* time, const float* x_spec,
                                          const dn_mesh_batch* batch, int64_t V, int K, int C, float* grad_x,
                                          float* grad_time, void* workspace, int64_t ws_bytes, int engine,
                                          dn_stream_t stream) {
  if (!grad_out || !mass || !evals || !evecs || !time || !x_spec || !grad_x || !grad_time || V < 0 || K <= 0 || C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  // grad_x = mass * (Phi_b dS_b) per tile: the from_basis chain with per-mesh weights and a row_scale epilogue
  DnLayer L = make_layer(nullptr, C, /*w_trans=*/1, nullptr, 0, K, C, grad_x, C);
  L.row_scale = mass;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc || (rc = grouped_spectral_check(grad_out, evecs, batch, V, K, C, tc, &L))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int64_t pb = tc_chain_ws_bytes(&L, 1) * batch->n_meshes;
  float* pk = ws.take(pb / 4);
  float* dt = ws.take(tc_spectral_bwd_batched_scratch_floats(batch->n_meshes, K, C));
  float* partial = ws.take((int64_t)batch->n_tb_ctas * K * C);
  if (!pk || !dt || !partial) return DN_ERR_WORKSPACE;
  // (nothing has been enqueued up to here)
  int P = 0;
  if ((rc = to_basis_tc(grad_out, evecs, nullptr, V, K, C, partial, &P, tc, st, batch))) return rc;
  if ((rc = tc_spectral_bwd_batched(&L, batch->n_meshes, pk, pb, partial, batch->mesh_cta_begin, evals, time, x_spec, dt,
                                    grad_time, batch->tile_mesh, st)))
    return rc;
  return tc_rows_chain(one_src(evecs, K, K), &L, 1, V, tc, ws.base + ws.off, ws.size - ws.off, st);
}

int dn_grad_spmm(const dn_csr* grad, const float* x, int64_t V, int C, float* out, dn_stream_t stream) {
  if (!grad || !grad->rowptr || !x || !out || V < 0 || C <= 0) return DN_ERR_INVALID_ARGUMENT;
  return launch_grad_spmm_pair(grad, x, V, C, out, (cudaStream_t)stream);
}

int dn_spatial_gradient_features_fwd(const float* vectors, const float* A_re, const float* A_im,
                                     int with_gradient_rotations, int64_t V, int C, float* out, void* workspace,
                                     int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!vectors || !A_re || (with_gradient_rotations && !A_im) || !out || V < 0 || C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  float* g01 = ws.take(V * 2 * C);
  float* b01 = ws.take(V * 2 * C);
  if (!g01 || !b01) return DN_ERR_WORKSPACE;
  int rc = launch_deinterleave_vc2(vectors, V, C, g01, st);
  if (rc) return rc;
  // Bre = g0 A_re^T - g1 A_im^T ; Bim = g1 A_re^T + g0 A_im^T   (layers.py:122-123)
  DnRowsSrc s0 = one_src(g01, C, 2 * C), s1 = one_src(g01 + C, C, 2 * C);
  if (with_gradient_rotations) {
    DnLayer T = make_layer(A_im, C, 0, nullptr, 0, C, C, b01, 2 * C);           // b0 = g1 A_im^T
    if ((rc = simt_rows_gemm(s1, T, V, st))) return rc;
    DnLayer L = make_layer(A_re, C, 0, nullptr, 0, C, C, b01, 2 * C);           // b0 = g0 A_re^T - b0
    L.residual = b01; L.ld_res = 2 * C; L.res_scale = -1.f;
    if ((rc = simt_rows_gemm(s0, L, V, st))) return rc;
    DnLayer M = make_layer(A_re, C, 0, nullptr, 0, C, C, b01 + C, 2 * C);       // b1 = g1 A_re^T
    if ((rc = simt_rows_gemm(s1, M, V, st))) return rc;
    DnLayer N2 = make_layer(A_im, C, 0, nullptr, 0, C, C, b01 + C, 2 * C);      // b1 = g0 A_im^T + b1
    N2.residual = b01 + C; N2.ld_res = 2 * C;
    if ((rc = simt_rows_gemm(s0, N2, V, st))) return rc;
  } else {
    DnLayer L = make_layer(A_re, C, 0, nullptr, 0, C, C, b01, 2 * C);           // layers.py:125-126
    if ((rc = simt_rows_gemm(s0, L, V, st))) return rc;
    L.out = b01 + C;
    if ((rc = simt_rows_gemm(s1, L, V, st))) return rc;
  }
  (void)engine;
  return launch_complex_dots_tanh(g01, b01, V, C, out, st);
}

int dn_gradient_features_fwd(const dn_csr* grad, const float* x_diffuse, const float* A_re, const float* A_im,
                             int with_gradient_rotations, int64_t V, int C, float* features, float* pq_out,
                             void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!grad || !grad->rowptr || !x_diffuse || !A_re || (with_gradient_rotations && !A_im) || !features || V < 0 ||
      C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  if (C % 4) return DN_ERR_UNSUPPORTED;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int npq = with_gradient_rotations ? 2 * C : C;
  float* pq = pq_out ? pq_out : ws.take(V * npq);
  if (!pq) return DN_ERR_WORKSPACE;
  DnRowsSrc src = one_src(x_diffuse, C, C);
  DnLayer L = make_layer(A_re, C, 0, nullptr, 0, C, npq, pq, npq);   // [P|Q] = xd [A_re;A_im]^T
  if (with_gradient_rotations) { L.W2 = A_im; L.n_split = C; }
  if ((rc = run_chain(src, &L, 1, V, tc, nullptr, nullptr, ws.base + ws.off, ws.size - ws.off, st))) return rc;
  return launch_spmm_features(grad, x_diffuse, pq, with_gradient_rotations, V, C, features, st);
}

int dn_gradient_features_bwd(const dn_csr* grad, const dn_csr* grad_t, const float* grad_features,
                             const float* x_diffuse, const float* pq, const float* features, const float* A_re,
                             const float* A_im, int with_gradient_rotations, int64_t V, int C, float* grad_x,
                             float* grad_A_re, float* grad_A_im, void* workspace, int64_t ws_bytes, int engine,
                             dn_stream_t stream) {
  if (!grad || !grad_t || !grad_features || !x_diffuse || !pq || !features || !A_re || !grad_x || !grad_A_re ||
      (with_gradient_rotations && (!A_im || !grad_A_im)))
    return DN_ERR_INVALID_ARGUMENT;
  if (C % 4) return DN_ERR_UNSUPPORTED;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int rot = with_gradient_rotations;
  float* U = ws.take(V * 4 * C);
  float* dxd = ws.take(V * C);
  float* dP = ws.take(V * C);                      // dP, dQ as two contiguous (V, C) matrices: they are the chain
  float* dQ = rot ? ws.take(V * C) : nullptr;      // kernel's two sources and the weight-gradient kernel's operands
  float* part = ws.take(kPartialFloats / 4);
  if (!U || !dxd || !dP || (rot && !dQ) || !part) return DN_ERR_WORKSPACE;
  void* tcws = ws.base + ws.off;
  const int64_t tcws_bytes = ws.size - ws.off;
  if ((rc = launch_features_bwd_local(grad, x_diffuse, pq, features, grad_features, rot, V, C, U, st))) return rc;
  if ((rc = launch_features_bwd_transpose(grad_t, U, rot, V, C, dxd, dP, dQ, C, st))) return rc;
  // grad_x = dxd + dP A_re (+ dQ A_im): one layer over the sources (dP | dQ) with [A_re ; A_im] stacked along K
  {
    DnRowsSrc s;
    memset(&s, 0, sizeof(s));
    s.ptr[0] = dP; s.width[0] = C; s.ld[0] = C; s.nsrc = 1;
    if (rot) { s.ptr[1] = dQ; s.width[1] = C; s.ld[1] = C; s.nsrc = 2; }
    DnLayer L = make_layer(A_re, C, /*w_trans=*/1, nullptr, 0, rot ? 2 * C : C, C, grad_x, C);
    if (rot) { L.W2 = A_im; L.n_split = C; }
    L.residual = dxd; L.ld_res = C;
    if (tc && tc_rows_chain_supported(s, &L, 1, tc) == DN_OK) {
      if ((rc = tc_rows_chain(s, &L, 1, V, tc, tcws, tcws_bytes, st))) return rc;
    } else {                                       // exact SIMT route: one source at a time
      if (tc && (rc = note_simt_fallback("a dense layer", L.K, L.N))) return rc;
      DnRowsSrc s0 = one_src(dP, C, C);
      DnLayer L0 = make_layer(A_re, C, 1, nullptr, 0, C, C, grad_x, C);
      L0.residual = dxd; L0.ld_res = C;
      if ((rc = simt_rows_gemm(s0, L0, V, st))) return rc;
      if (rot) {
        DnRowsSrc s1 = one_src(dQ, C, C);
        DnLayer L1 = make_layer(A_im, C, 1, nullptr, 0, C, C, grad_x, C);
        L1.residual = grad_x; L1.ld_res = C;
        if ((rc = simt_rows_gemm(s1, L1, V, st))) return rc;
      }
    }
  }
  // grad_A_re[n][k] += sum_v dP[v][n] xd[v][k]   (and grad_A_im from dQ)
  if ((rc = atb(dP, C, C, x_diffuse, C, C, V, grad_A_re, C, 1, part, kPartialFloats / 4, tc, st))) return rc;
  if (rot)
    if ((rc = atb(dQ, C, C, x_diffuse, C, C, V, grad_A_im, C, 1, part, kPartialFloats / 4, tc, st))) return rc;
  return DN_OK;
}

int dn_mini_mlp_fwd(const float* const* src_host, const int* src_width_host, int nsrc,
                    const float* const* weight_host, const float* const* bias_host, const int* dims_host,
                    int n_layers, const float* const* drop_mask_host, const float* residual, int64_t V,
                    float* const* hidden_out_host, float* out, void* workspace, int64_t ws_bytes, int engine,
                    dn_stream_t stream) {
  if (!src_host || !src_width_host || nsrc < 1 || nsrc > DN_MAX_SRC || !weight_host || !dims_host || n_layers < 1 ||
      n_layers > DN_MAX_LAYERS || !out || V < 0)
    return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  DnRowsSrc src;
  memset(&src, 0, sizeof(src));
  int k0 = 0;
  for (int s = 0; s < nsrc; ++s) {
    if (!src_host[s] || src_width_host[s] <= 0) return DN_ERR_INVALID_ARGUMENT;
    src.ptr[s] = src_host[s]; src.width[s] = src_width_host[s]; src.ld[s] = src_width_host[s];
    k0 += src_width_host[s];
  }
  src.nsrc = nsrc;
  if (k0 != dims_host[0]) return DN_ERR_INVALID_ARGUMENT;
  DnLayer layers[DN_MAX_LAYERS];
  int maxn = 0;
  for (int l = 0; l < n_layers; ++l) {
    if (!weight_host[l] || dims_host[l + 1] <= 0) return DN_ERR_INVALID_ARGUMENT;
    const bool last = (l + 1 == n_layers);
    float* o = last ? out : (hidden_out_host ? hidden_out_host[l] : nullptr);
    layers[l] = make_layer(weight_host[l], dims_host[l], 0, bias_host ? bias_host[l] : nullptr, last ? 0 : 1,
                           dims_host[l], dims_host[l + 1], o, dims_host[l + 1]);
    if (!last && drop_mask_host) layers[l].emul = drop_mask_host[l];
    if (last && residual) { layers[l].residual = residual; layers[l].ld_res = dims_host[l + 1]; }
    if (dims_host[l + 1] > maxn) maxn = dims_host[l + 1];
  }
  Bump ws(workspace, ws_bytes);
  float *t0 = nullptr, *t1 = nullptr;
  const bool fused = tc && tc_rows_chain_supported(src, layers, n_layers, tc) == DN_OK;
  if (!fused && n_layers > 1) {
    t0 = ws.take(V * maxn);
    t1 = ws.take(V * maxn);
    if (!t0 || !t1) return DN_ERR_WORKSPACE;
  }
  return run_chain(src, layers, n_layers, V, tc, t0, t1, ws.base + ws.off, ws.size - ws.off, (cudaStream_t)stream);
}

int dn_mini_mlp_bwd(const float* grad_out, const float* const* src_host, const int* src_width_host, int nsrc,
                    const float* const* weight_host, const int* dims_host, int n_layers,
                    const float* const* hidden_host, const float* const* drop_mask_host, int64_t V,
                    float* const* grad_src_host, float* const* grad_weight_host, float* const* grad_bias_host,
                    void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!grad_out || !src_host || !src_width_host || nsrc < 1 || nsrc > DN_MAX_SRC || !weight_host || !dims_host ||
      n_layers < 1 || n_layers > DN_MAX_LAYERS || (n_layers > 1 && !hidden_host) || !grad_src_host ||
      !grad_weight_host)
    return DN_ERR_INVALID_ARGUMENT;
  int tc, rc = resolve_engine(engine, &tc);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  int maxn = 0;
  for (int l = 0; l <= n_layers; ++l) maxn = dims_host[l] > maxn ? dims_host[l] : maxn;
  Bump ws(workspace, ws_bytes);
  float* d0 = ws.take(V * maxn);
  float* d1 = ws.take(V * maxn);
  float* part = ws.take(kPartialFloats / 2);
  if (!d0 || !d1 || !part) return DN_ERR_WORKSPACE;
  void* tcws = ws.base + ws.off;
  const int64_t tcws_bytes = ws.size - ws.off;
  const float* dz = grad_out;   // gradient w.r.t. the pre-activation of layer l
  for (int l = n_layers - 1; l >= 0; --l) {
    const int nout = dims_host[l + 1], nin = dims_host[l];
    // weight / bias gradients:  grad_W[n][k] += sum_v dz[v][n] * h_{l-1}[v][k]
    if (l > 0) {
      if ((rc = atb(dz, nout, nout, hidden_host[l - 1], nin, nin, V, grad_weight_host[l], nin, 1, part,
                    kPartialFloats / 2, tc, st)))
        return rc;
    } else {
      int off = 0;
      for (int s = 0; s < nsrc; ++s) {
        if ((rc = atb(dz, nout, nout, src_host[s], src_width_host[s], src_width_host[s], V, grad_weight_host[0] + off,
                      nin, 1, part, kPartialFloats / 2, tc, st)))
          return rc;
        off += src_width_host[s];
      }
    }
    if (grad_bias_host && grad_bias_host[l])
      if ((rc = simt_colsum(dz, nout, nout, V, grad_bias_host[l], 1, st))) return rc;
    // input gradient:  dz_{l-1} = (dz_l W_l) * 1[h_{l-1} > 0] (* dropout mask)
    DnRowsSrc s = one_src(dz, nout, nout);
    if (l > 0) {
      float* o = (dz == d0) ? d1 : d0;
      DnLayer L = make_layer(weight_host[l], nin, /*w_trans=*/1, nullptr, 0, nout, nin, o, nin);
      L.relu_mask_src = hidden_host[l - 1];
      if (drop_mask_host && drop_mask_host[l - 1]) L.emul = drop_mask_host[l - 1];
      if ((rc = run_chain(s, &L, 1, V, tc, nullptr, nullptr, tcws, tcws_bytes, st))) return rc;
      dz = o;
    } else {
      int off = 0;
      for (int q = 0; q < nsrc; ++q) {
        if (grad_src_host[q]) {
          DnLayer L = make_layer(weight_host[0] + off, nin, 1, nullptr, 0, nout, src_width_host[q], grad_src_host[q],
                                 src_width_host[q]);
          if ((rc = run_chain(s, &L, 1, V, tc, nullptr, nullptr, tcws, tcws_bytes, st))) return rc;
        }
        off += src_width_host[q];
      }
    }
  }
  return DN_OK;
}

static int block_fwd_impl(const float* x_in, const float* mass, const float* evals, const float* evecs,
                          const dn_csr* grad, const dn_block_params* p, int64_t V, int K, int C, float* out,
                          void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream, cudaEvent_t* ev,
                          const dn_mesh_batch* batch = nullptr, const dn_head* head = nullptr) {
  // ev (optional, DN_PROFILE_STAGES + 1 events): recorded on the launching stream between the stages
  auto mark = [&](int i) { if (ev) cudaEventRecord(ev[i], (cudaStream_t)stream); };
  if (!x_in || !mass || !evals || !evecs || !p || !p->diffusion_time || (!out && !head) || V < 0 || K <= 0 || C <= 0)
    return DN_ERR_INVALID_ARGUMENT;
  if (head && (!head->weight || !head->out || head->n_out < 1 || head->n_out > 8 || head->ld_out < head->n_out))
    return DN_ERR_INVALID_ARGUMENT;
  if (p->with_gradient_features && (!grad || !grad->rowptr || !p->A_re || (p->with_gradient_rotations && !p->A_im)))
    return DN_ERR_INVALID_ARGUMENT;
  if (p->n_mlp_layers < 1 || p->n_mlp_layers > DN_MAX_LAYERS || !p->mlp_weight_host || !p->mlp_dims_host)
    return DN_ERR_INVALID_ARGUMENT;
  if (p->with_gradient_features && (C % 4)) return DN_ERR_UNSUPPORTED;
  int tc, rc = resolve_engine(engine, &tc), P = 0;
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  Bump ws(workspace, ws_bytes);
  const int rot = p->with_gradient_rotations;
  const int npq = rot ? 2 * C : C;
  float* S = ws.take((int64_t)K * C);
  float* xd = ws.take(V * C);
  float* pq = p->with_gradient_features ? ws.take(V * npq) : nullptr;
  float* feat = p->with_gradient_features ? ws.take(V * C) : nullptr;
  const int64_t pf = kPartialFloats;
  float* partial = ws.take(pf);
  if (!S || !xd || !partial || (p->with_gradient_features && (!pq || !feat))) return DN_ERR_WORKSPACE;

  // every dense layer of the block: [0] from_basis, [1] (a5, commuted) [P|Q] = x_diffuse [A_re;A_im]^T,
  // [2..] cat -> MiniMLP -> + x_in  [layers.py:229-239]
  const int nm = p->n_mlp_layers;
  DnLayer L[3 + DN_MAX_LAYERS];
  L[0] = make_layer(S, C, 1, nullptr, 0, K, C, xd, C);
  int nfront = 1;
  // Tensor-core gradient features (C_width = 128, learned rotations, fp32-grade / TF32 engines): gather only x_diffuse
  // (gxy = [gradX x | gradY x], a third of the commuted route's gather traffic), then the complex-linear map as tcgen05
  // GEMMs whose epilogue forms tanh(gX * Bre + gY * Bim) (layers.py:117-130) -- two launches of 64 channels each, so
  // that the [Bre | Bim] accumulators (128 columns) ping-pong in TMEM.  Every other block takes the commuted route
  // ([P|Q] = x_diffuse [A_re; A_im]^T in front of a gather of x, P and Q).
  bool gf_tc = false;
  DnRowsSrc src_gxy = one_src(pq, 2 * C, 2 * C);
  if (p->with_gradient_features && rot && C == 128 && tc && tc != DN_PASSES_BF16 &&
      !(grad->patches && grad->patches->n_patches > 0)) {
    for (int h = 0; h < 2; ++h) {
      L[1 + h] = make_layer(p->A_re, C, 0, nullptr, 0, 2 * C, C, feat + h * 64, C);
      L[1 + h].W2 = p->A_im; L[1 + h].rot_C = C; L[1 + h].rot_ch0 = h * 64;
      L[1 + h].dots_src = pq + h * 64; L[1 + h].ld_dots = 2 * C; L[1 + h].dots_gy_col = C;
    }
    gf_tc = tc_rows_chain_supported(src_gxy, &L[1], 1, tc) == DN_OK &&
            tc_rows_chain_supported(src_gxy, &L[2], 1, tc) == DN_OK;
    if (gf_tc) nfront = 3;
  }
  if (p->with_gradient_features && !gf_tc) {
    if (rot && npq > 256) {
      // [P|Q] wider than one tensor-core layer (C_width = 256): P and Q are separate layers writing the two halves
      L[1] = make_layer(p->A_re, C, 0, nullptr, 0, C, C, pq, npq);
      L[2] = make_layer(p->A_im, C, 0, nullptr, 0, C, C, pq + C, npq);
      nfront = 3;
    } else {
      L[1] = make_layer(p->A_re, C, 0, nullptr, 0, C, npq, pq, npq);
      if (rot) { L[1].W2 = p->A_im; L[1].n_split = C; }
      nfront = 2;
    }
  }
  const int nsrc = p->with_gradient_features ? 3 : 2;
  if (p->mlp_dims_host[0] != nsrc * C) return DN_ERR_INVALID_ARGUMENT;
  int maxn = 0;
  for (int l = 0; l < nm; ++l) {
    const bool last = (l + 1 == nm);
    if (!p->mlp_weight_host[l] || p->mlp_dims_host[l + 1] <= 0) return DN_ERR_INVALID_ARGUMENT;
    L[nfront + l] = make_layer(p->mlp_weight_host[l], p->mlp_dims_host[l], 0,
                               p->mlp_bias_host ? p->mlp_bias_host[l] : nullptr, last ? 0 : 1, p->mlp_dims_host[l],
                               p->mlp_dims_host[l + 1], last ? out : nullptr, p->mlp_dims_host[l + 1]);
    if (last) {
      L[nfront + l].residual = x_in; L[nfront + l].ld_res = C;
      if (head) {        // DiffusionNet.last_lin in this layer's epilogue; the block output itself is not stored
        DnLayer& Lh = L[nfront + l];
        Lh.head_w = head->weight; Lh.head_b = head->bias; Lh.head_out = head->out; Lh.ld_head_out = head->ld_out;
        Lh.head_n = head->n_out;
        if (!out) Lh.out = nullptr;
      }
    }
    if (p->mlp_dims_host[l + 1] > maxn) maxn = p->mlp_dims_host[l + 1];
  }
  if (p->mlp_dims_host[nm] != C) return DN_ERR_INVALID_ARGUMENT;
  DnRowsSrc src_fb = one_src(evecs, K, K);
  DnRowsSrc src_pq = one_src(xd, C, C);
  DnRowsSrc src_mlp;
  memset(&src_mlp, 0, sizeof(src_mlp));
  const float* srcs[3] = {x_in, xd, feat};
  for (int q = 0; q < nsrc; ++q) { src_mlp.ptr[q] = srcs[q]; src_mlp.width[q] = C; src_mlp.ld[q] = C; }
  src_mlp.nsrc = nsrc;
  // one launch packs (hi/lo split + UMMA layout) every weight the tensor-core kernels will stream
  const bool front_fused = tc && nfront == 2 && tc_rows_chain_supported(src_fb, &L[0], 2, tc) == DN_OK;
  bool tc_front = front_fused;
  const DnRowsSrc& src_l12 = gf_tc ? src_gxy : src_pq;      // input of L[1], L[2]: raw gradients | x_diffuse
  if (tc && !front_fused) {
    tc_front = tc_rows_chain_supported(src_fb, &L[0], 1, tc) == DN_OK;
    for (int l = 1; l < nfront; ++l) tc_front = tc_front && tc_rows_chain_supported(src_l12, &L[l], 1, tc) == DN_OK;
  }
  if (gf_tc && !tc_front) return DN_ERR_UNSUPPORTED;         // (from_basis outside the envelope: cannot happen at C = 128)
  const bool tc_mlp = tc && tc_rows_chain_supported(src_mlp, &L[nfront], nm, tc) == DN_OK;
  if (head && !tc_mlp) return DN_ERR_UNSUPPORTED;
  // the spectral multiplier S = exp(-lambda t) * (reduced partial sums) is layer 0's weight: when the tensor-core path
  // takes the front chain it is formed inside the pack launch (no separate scale kernel, S never round-trips HBM)
  if (batch) {
    if ((rc = check_batch(batch, x_in, evecs, V, K, C))) return rc;
    if (!tc_front || (int64_t)batch->n_tb_ctas * K * C > pf) return DN_ERR_UNSUPPORTED;
  }
  // (nothing has been launched up to here: an unsupported head / batch returns before any work is enqueued)
  mark(0);
  // (a1) spectral diffusion: to_basis -> exp(-lambda t) -> from_basis   [layers.py:56-67]; over a batch the grouped
  // split-V to_basis, every CTA reducing a row range inside one mesh
  if (batch) {
    if ((rc = to_basis_tc(x_in, evecs, mass, V, K, C, partial, &P, tc, st, batch))) return rc;
  } else if ((rc = to_basis_partials(x_in, evecs, mass, V, K, C, partial, pf, &P, tc, st))) {
    return rc;
  }
  mark(1);
  if (!tc_front)
    if ((rc = launch_spectral_scale(partial, P, evals, p->diffusion_time, K, C, nullptr, S, 1, st))) return rc;
  mark(2);
  if (tc_front) {
    if (front_fused) tc_choose_pack_fmt(src_fb, &L[0], 2, tc);
    else {
      tc_choose_pack_fmt(src_fb, &L[0], 1, tc);
      for (int l = 1; l < nfront; ++l) tc_choose_pack_fmt(src_l12, &L[l], 1, tc);
    }
  }
  if (tc_mlp) tc_choose_pack_fmt(src_mlp, &L[nfront], nm, tc);
  if (batch) {
    // one packed spectral multiplier per mesh (layer 0 of the front chain picks its matrix per tile), then every other
    // weight of the block in one more launch
    const int64_t pb0 = tc_chain_ws_bytes(&L[0], 1) * batch->n_meshes;
    float* pk0 = ws.take(pb0 / 4);
    if (!pk0) return DN_ERR_WORKSPACE;
    if ((rc = tc_pack_spectral_batched(&L[0], batch->n_meshes, pk0, pb0, partial, batch->mesh_cta_begin, evals,
                                       p->diffusion_time, 1, batch->tile_mesh, st)))
      return rc;
    const int cnt = (nfront - 1) + (tc_mlp ? nm : 0);
    if (cnt > 0) {
      DnLayer* first = (nfront > 1) ? &L[1] : &L[nfront];
      const int64_t pb = tc_chain_ws_bytes(first, cnt);
      float* pk = ws.take(pb / 4);
      if (!pk) return DN_ERR_WORKSPACE;
      if ((rc = tc_pack_layers(first, cnt, pk, pb, st))) return rc;
    }
  } else if (tc_front || tc_mlp) {
    DnLayer* first = tc_front ? &L[0] : &L[nfront];
    const int cnt = (tc_front ? nfront : 0) + (tc_mlp ? nm : 0);
    const int64_t pb = tc_chain_ws_bytes(first, cnt);
    float* pk = ws.take(pb / 4);
    if (!pk) return DN_ERR_WORKSPACE;
    if (tc_front) rc = tc_pack_layers_spectral(first, cnt, pk, pb, partial, P, evals, p->diffusion_time, 1, st);
    else rc = tc_pack_layers(first, cnt, pk, pb, st);
    if (rc) return rc;
  }
  mark(3);
  float *t0 = nullptr, *t1 = nullptr;
  if (!tc_mlp && nm > 1) {
    t0 = ws.take(V * maxn);
    t1 = ws.take(V * maxn);
    if (!t0 || !t1) return DN_ERR_WORKSPACE;
  }
  void* tcws = ws.base + ws.off;
  const int64_t tcws_bytes = ws.size - ws.off;
  // from_basis and [P|Q]: one fused two-layer chain when it fits, else one launch per layer
  if (front_fused) {
    if ((rc = run_chain(src_fb, &L[0], 2, V, tc, nullptr, nullptr, tcws, tcws_bytes, st))) return rc;
  } else {
    if ((rc = run_chain(src_fb, &L[0], 1, V, tc, nullptr, nullptr, tcws, tcws_bytes, st))) return rc;
    if (!gf_tc)
      for (int l = 1; l < nfront; ++l)
        if ((rc = run_chain(src_pq, &L[l], 1, V, tc, nullptr, nullptr, tcws, tcws_bytes, st))) return rc;
  }
  mark(4);
  // (a4+a5) sparse tangent gradient + complex inner product + tanh   [layers.py:216-226,128-130]
  if (gf_tc) {
    if ((rc = launch_spmm_gxy(grad, xd, V, C, pq, st))) return rc;
    if (ev) {
      if (!g_gf_ev) cudaEventCreate(&g_gf_ev);
      if (g_gf_ev) { cudaEventRecord(g_gf_ev, st); g_gf_recorded = true; }
    }
    for (int l = 1; l < nfront; ++l)
      if ((rc = tc_rows_chain(src_gxy, &L[l], 1, V, tc, tcws, tcws_bytes, st))) return rc;
  } else if (p->with_gradient_features) {
    if ((rc = launch_spmm_features(grad, xd, pq, rot, V, C, feat, st))) return rc;
  }
  mark(5);
  rc = run_chain(src_mlp, &L[nfront], nm, V, tc, t0, t1, tcws, tcws_bytes, st);
  mark(6);
  return rc;
}

int dn_block_fwd(const float* x_in, const float* mass, const float* evals, const float* evecs, const dn_csr* grad,
                 const dn_block_params* p, int64_t V, int K, int C, float* out, void* workspace, int64_t ws_bytes,
                 int engine, dn_stream_t stream) {
  return block_fwd_impl(x_in, mass, evals, evecs, grad, p, V, K, C, out, workspace, ws_bytes, engine, stream, nullptr);
}

int dn_block_fwd_batched(const float* x_in, const float* mass, const float* evals, const float* evecs, const dn_csr* grad,
                         const dn_block_params* p, const dn_mesh_batch* batch, int64_t V, int K, int C, float* out,
                         void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  if (!batch) return DN_ERR_INVALID_ARGUMENT;
  return block_fwd_impl(x_in, mass, evals, evecs, grad, p, V, K, C, out, workspace, ws_bytes, engine, stream, nullptr, batch);
}

int dn_block_fwd_ex(const float* x_in, const float* mass, const float* evals, const float* evecs, const dn_csr* grad,
                    const dn_block_params* p, const dn_mesh_batch* batch, const dn_head* head, int64_t V, int K, int C,
                    float* out, void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream) {
  return block_fwd_impl(x_in, mass, evals, evecs, grad, p, V, K, C, out, workspace, ws_bytes, engine, stream, nullptr, batch, head);
}

int dn_mesh_batch_plan(int n_meshes, const int32_t* n_rows_host, int sm_count, int32_t* row_begin_host,
                       int32_t* tile_mesh_host, int32_t* tb_rows_host, int32_t* mesh_cta_begin_host) {
  if (n_meshes < 1 || !n_rows_host || !row_begin_host || !tile_mesh_host || !tb_rows_host || !mesh_cta_begin_host)
    return DN_ERR_INVALID_ARGUMENT;
  if (sm_count < 1) sm_count = 148;
  int64_t row = 0, chunks_total = 0;
  for (int b = 0; b < n_meshes; ++b) {
    if (n_rows_host[b] < 0) return DN_ERR_INVALID_ARGUMENT;
    row_begin_host[b] = (int32_t)row;
    const int64_t padded = ((int64_t)n_rows_host[b] + 127) / 128 * 128;
    for (int64_t t = row / 128; t < (row + padded) / 128; ++t) tile_mesh_host[t] = b;
    row += padded;
    if (row >= (1ll << 31) - 256) return DN_ERR_UNSUPPORTED;
    chunks_total += ((int64_t)n_rows_host[b] + 15) / 16;
  }
  row_begin_host[n_meshes] = (int32_t)row;
  // CTAs per mesh proportional to its 16-row chunks (>= 1), about sm_count in total, at most 1024
  int n_ctas = 0;
  for (int b = 0; b < n_meshes; ++b) {
    const int64_t chunks = ((int64_t)n_rows_host[b] + 15) / 16;
    int64_t want = chunks_total > 0 ? (chunks * sm_count + chunks_total / 2) / chunks_total : 1;
    if (want < 1) want = 1;
    if (want > chunks && chunks > 0) want = chunks;
    if (n_ctas + want + (n_meshes - 1 - b) > 1024) want = 1;
    if (n_ctas + want > 1024) return DN_ERR_UNSUPPORTED;
    mesh_cta_begin_host[b] = n_ctas;
    const int64_t per = chunks > 0 ? (chunks + want - 1) / want : 0;
    if (per > 0) want = (chunks + per - 1) / per;              // no empty CTAs
    for (int64_t c = 0; c < want; ++c) {
      int64_t rb = row_begin_host[b] + c * per * 16;
      int64_t re = rb + per * 16;
      const int64_t end = (int64_t)row_begin_host[b] + n_rows_host[b];
      if (rb > end) rb = end;
      if (re > end) re = end;
      tb_rows_host[2 * n_ctas] = (int32_t)rb;
      tb_rows_host[2 * n_ctas + 1] = (int32_t)re;
      ++n_ctas;
    }
  }
  mesh_cta_begin_host[n_meshes] = n_ctas;
  return n_ctas;
}

int dn_block_fwd_profile(const float* x_in, const float* mass, const float* evals, const float* evecs,
                         const dn_csr* grad, const dn_block_params* p, int64_t V, int K, int C, float* out,
                         void* workspace, int64_t ws_bytes, int engine, dn_stream_t stream, float* stage_ms_host) {
  if (!stage_ms_host) return DN_ERR_INVALID_ARGUMENT;
  cudaEvent_t ev[DN_PROFILE_STAGES + 1];
  g_gf_recorded = false;
  g_gf_gather_ms = 0.f;
  for (int i = 0; i <= DN_PROFILE_STAGES; ++i) DN_CUDA_TRY(cudaEventCreate(&ev[i]));
  int rc = block_fwd_impl(x_in, mass, evals, evecs, grad, p, V, K, C, out, workspace, ws_bytes, engine, stream, ev);
  if (rc == DN_OK) {
    rc = (int)cudaEventSynchronize(ev[DN_PROFILE_STAGES]);
    for (int i = 0; i < DN_PROFILE_STAGES && rc == DN_OK; ++i)
      rc = (int)cudaEventElapsedTime(&stage_ms_host[i], ev[i], ev[i + 1]);
    if (rc == DN_OK && g_gf_recorded && cudaEventElapsedTime(&g_gf_gather_ms, ev[4], g_gf_ev) != cudaSuccess) cudaGetLastError();
  }
  for (int i = 0; i <= DN_PROFILE_STAGES; ++i) cudaEventDestroy(ev[i]);
  return rc;
}

}  // extern "C"
