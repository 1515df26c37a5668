// SIMT (FFMA, exact fp32) kernels of the DiffusionNetBlock hot path, and the sparse /
// elementwise kernels shared by every engine.  sm_100a only.
//
// Reference functions restated here (file:line in /root/reference/src/diffusion_net):
//   to_basis geometry.py:572-583, from_basis geometry.py:586-598,
//   LearnedTimeDiffusion.forward layers.py:44-67, grad SpMM layers.py:216-223,
//   SpatialGradientFeatures.forward layers.py:117-130, MiniMLP layers.py:133-164.
#include "dn_internal.h"
#include "dn_tc_ptx.cuh"
#include <math.h>

namespace {

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// ---------------------------------------------------------------------------------------------
// rows GEMM:  out[v][n] = epi( sum_k A[v][k] * W[n][k] + bias[n] ),  A = concat of up to 3 sources
// ---------------------------------------------------------------------------------------------
constexpr int RG_BM = 128, RG_BN = 64, RG_BK = 16;

__device__ __forceinline__ float load_src_scalar(const DnRowsSrc& s, int64_t row, int k) {
#pragma unroll
  for (int i = 0; i < DN_MAX_SRC; ++i) {
    if (i < s.nsrc) {
      if (k < s.width[i]) return __ldg(s.ptr[i] + row * s.ld[i] + k);
      k -= s.width[i];
    }
  }
  return 0.f;
}

__device__ __forceinline__ float4 load_src_vec4(const DnRowsSrc& s, int64_t row, int k) {
#pragma unroll
  for (int i = 0; i < DN_MAX_SRC; ++i) {
    if (i < s.nsrc) {
      if (k < s.width[i]) return ldg4(s.ptr[i] + row * s.ld[i] + k);
      k -= s.width[i];
    }
  }
  return make_float4(0.f, 0.f, 0.f, 0.f);
}

template <bool VEC>
__global__ void __launch_bounds__(256) rows_gemm_kernel(DnRowsSrc src, DnLayer L, int64_t V) {
  __shared__ __align__(16) float As[RG_BK][RG_BM + 4];
  __shared__ __align__(16) float Bs[RG_BK][RG_BN + 4];
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t row0 = (int64_t)blockIdx.x * RG_BM;
  const int n0 = blockIdx.y * RG_BN;
  const int K = L.K, N = L.N;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int k0 = 0; k0 < K; k0 += RG_BK) {
    // ---- A tile: 128 rows x 16 k, transposed into As[k][row]
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      const int r = (t >> 2) + 64 * i;
      const int kq = (t & 3) * 4;
      const int64_t gr = row0 + r;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (gr < V) {
        if (VEC && k0 + kq + 3 < K) {
          float4 q = load_src_vec4(src, gr, k0 + kq);
          v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (k0 + kq + j < K) v[j] = load_src_scalar(src, gr, k0 + kq + j);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) As[kq + j][r] = v[j];
    }
    // ---- B tile: 16 k x 64 n into Bs[k][n]
    if (!L.w_trans) {
      const int n = t >> 2, kq = (t & 3) * 4, gn = n0 + n;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (gn < N) {
        const float* wp = (L.W2 && gn >= L.n_split) ? L.W2 + (int64_t)(gn - L.n_split) * L.ldw + k0 + kq
                                                    : L.W + (int64_t)gn * L.ldw + k0 + kq;
        if (VEC && k0 + kq + 3 < K) {
          float4 q = ldg4(wp);
          v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (k0 + kq + j < K) v[j] = __ldg(wp + j);
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) Bs[kq + j][n] = v[j];
    } else {
      const int k = t >> 4, nq = (t & 15) * 4;
      float v[4] = {0.f, 0.f, 0.f, 0.f};
      if (k0 + k < K) {
        const float* wp = L.W + (int64_t)(k0 + k) * L.ldw + n0 + nq;
        if (VEC && n0 + nq + 3 < N) {
          float4 q = ldg4(wp);
          v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n0 + nq + j < N) v[j] = __ldg(wp + j);
        }
      }
      *reinterpret_cast<float4*>(&Bs[k][nq]) = make_float4(v[0], v[1], v[2], v[3]);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < RG_BK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  // ---- epilogue
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t gr = row0 + ty * 8 + i;
    if (gr >= V) continue;
    const float rs = L.row_scale ? __ldg(L.row_scale + gr) : 1.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn >= N) continue;
      float v = acc[i][j];
      if (L.bias) v += __ldg(L.bias + gn);
      if (L.relu) v = fmaxf(v, 0.f);
      if (L.emul) v *= __ldg(L.emul + gr * N + gn);
      if (L.relu_mask_src) v = (__ldg(L.relu_mask_src + gr * N + gn) > 0.f) ? v : 0.f;
      if (L.row_scale) v *= rs;
      if (L.residual) v = fmaf(L.res_scale, L.residual[gr * L.ld_res + gn], v);
      L.out[gr * L.ld_out + gn] = v;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// A^T B with a long reduction over vertices (to_basis, weight gradients):
//   partial[p][i][j] = sum_{v in split p} A[v][i] * scale[v] * B[v][j]
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) atb_partial_kernel(const float* __restrict__ A, int64_t lda, int I,
                                                          const float* __restrict__ B, int64_t ldb, int J,
                                                          const float* __restrict__ scale, int64_t V,
                                                          int64_t rows_per_split, float* __restrict__ partial) {
  __shared__ __align__(16) float As[16][64 + 4];
  __shared__ __align__(16) float Bs[16][64 + 4];
  const int tilesJ = (J + 63) / 64;
  const int i0 = (blockIdx.x / tilesJ) * 64, j0 = (blockIdx.x % tilesJ) * 64;
  const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
  const int64_t vbeg = (int64_t)blockIdx.y * rows_per_split;
  const int64_t vend = min(V, vbeg + rows_per_split);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const bool veca = ((lda & 3) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
  const bool vecb = ((ldb & 3) == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
  for (int64_t v0 = vbeg; v0 < vend; v0 += 16) {
    const int r = t >> 4, c4 = (t & 15) * 4;
    const int64_t gv = v0 + r;
    float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
    if (gv < vend) {
      const float s = scale ? __ldg(scale + gv) : 1.f;
      if (veca && i0 + c4 + 3 < I) {
        float4 q = ldg4(A + gv * lda + i0 + c4);
        a[0] = q.x; a[1] = q.y; a[2] = q.z; a[3] = q.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (i0 + c4 + j < I) a[j] = __ldg(A + gv * lda + i0 + c4 + j);
      }
      if (vecb && j0 + c4 + 3 < J) {
        float4 q = ldg4(B + gv * ldb + j0 + c4);
        b[0] = q.x; b[1] = q.y; b[2] = q.z; b[3] = q.w;
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j0 + c4 + j < J) b[j] = __ldg(B + gv * ldb + j0 + c4 + j);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] *= s;   // (values * massvec) as in geometry.py:583
    }
    *reinterpret_cast<float4*>(&As[r][c4]) = make_float4(a[0], a[1], a[2], a[3]);
    *reinterpret_cast<float4*>(&Bs[r][c4]) = make_float4(b[0], b[1], b[2], b[3]);
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float aa[4] = {av.x, av.y, av.z, av.w};
      const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(aa[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* pp = partial + (int64_t)blockIdx.y * I * J;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = i0 + ty * 4 + i;
    if (gi >= I) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gj = j0 + tx * 4 + j;
      if (gj < J) pp[(int64_t)gi * J + gj] = acc[i][j];
    }
  }
}

__global__ void reduce_partials_ld_kernel(const float* __restrict__ partial, int P, int I, int J,
                                          float* __restrict__ out, int64_t ld_out, int accumulate) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)I * J) return;
  float s = 0.f;
  for (int p = 0; p < P; ++p) s += partial[(int64_t)p * I * J + idx];
  const int i = (int)(idx / J), j = (int)(idx % J);
  float* o = out + (int64_t)i * ld_out + j;
  *o = accumulate ? (*o + s) : s;
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, int P, int64_t n, float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  float s = 0.f;
  for (int p = 0; p < P; ++p) s += partial[(int64_t)p * n + idx];
  out[idx] = s;
}

__global__ void colsum_kernel(const float* __restrict__ A, int64_t lda, int N, int64_t V, float* __restrict__ out) {
  // block (32, 8): 256 rows per block, 32 columns
  __shared__ float red[8][33];
  const int n = blockIdx.y * 32 + threadIdx.x;
  const int64_t v0 = (int64_t)blockIdx.x * 256;
  float s = 0.f;
  if (n < N)
    for (int r = threadIdx.y; r < 256; r += 8) {
      const int64_t v = v0 + r;
      if (v < V) s += __ldg(A + v * lda + n);
    }
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float tot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) tot += red[i][threadIdx.x];
    atomicAdd(out + n, tot);
  }
}

// ---------------------------------------------------------------------------------------------
// spectral coefficient kernels (layers.py:48-49, 62-64)
// ---------------------------------------------------------------------------------------------
__global__ void spectral_scale_kernel(const float* __restrict__ partial, int P, const float* __restrict__ evals,
                                      float* __restrict__ time, int K, int C, float* __restrict__ x_spec_out,
                                      float* __restrict__ S_out, int clamp_writeback) {
  // block = 64 consecutive elements x 4 slices of the P partial sums (more loads in flight)
  __shared__ float red[4][64];
  const int e = threadIdx.x & 63, sl = threadIdx.x >> 6;
  const int idx = blockIdx.x * 64 + e;
  float acc = 0.f;
  if (idx < K * C)
    for (int p = sl; p < P; p += 4) acc += partial[(int64_t)p * K * C + idx];
  red[sl][e] = acc;
  __syncthreads();
  if (sl != 0 || idx >= K * C) return;
  const int k = idx / C, c = idx % C;
  const float s = (red[0][e] + red[1][e]) + (red[2][e] + red[3][e]);
  const float t = fmaxf(time[c], 1e-8f);              // torch.clamp(t, min=1e-8)
  const float coef = expf(-(evals[k] * t));           // torch.exp(-evals.unsqueeze(-1) * time.unsqueeze(0))
  if (x_spec_out) x_spec_out[idx] = s;
  S_out[idx] = coef * s;
  // every thread of row k == 0 re-writes the clamped time (same value from all writers is benign)
  if (clamp_writeback && k == K - 1) {
    // last row, after all reads of time[c] by this thread; other threads read the same c only
    // through fmaxf(...,1e-8) which is idempotent under this write.
    time[c] = t;
  }
}

// backward: Gs = sum_p partial (= Phi^T g), dS = E * Gs, dt[c] += sum_k Gs*( -lambda_k )*E*x_spec
__global__ void spectral_bwd_kernel(const float* __restrict__ partial, int P, const float* __restrict__ evals,
                                    const float* __restrict__ time, const float* __restrict__ x_spec, int K, int C,
                                    float* __restrict__ dS, float* __restrict__ grad_time) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float t = fmaxf(time[c], 1e-8f);
  float dt = 0.f;
  for (int k = 0; k < K; ++k) {
    const int idx = k * C + c;
    float g = 0.f;
    for (int p = 0; p < P; ++p) g += partial[(int64_t)p * K * C + idx];
    const float lam = evals[k];
    const float e = expf(-(lam * t));
    dS[idx] = e * g;
    dt += g * (-lam) * e * x_spec[idx];
  }
  grad_time[c] += dt;
}

// ---------------------------------------------------------------------------------------------
// sparse kernels
// ---------------------------------------------------------------------------------------------
__global__ void csr_from_coo_kernel(const int64_t* __restrict__ rows, const int64_t* __restrict__ cols,
                                    const float* __restrict__ vx, const float* __restrict__ vy, int64_t nnz,
                                    int64_t V, int32_t* __restrict__ rowptr, int32_t* __restrict__ colidx,
                                    float* __restrict__ vals) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nnz) return;
  const int64_t r = rows[p];
  const int64_t rprev = (p == 0) ? -1 : rows[p - 1];
  for (int64_t rr = rprev + 1; rr <= r; ++rr) rowptr[rr] = (int32_t)p;
  if (p == nnz - 1)
    for (int64_t rr = r + 1; rr <= V; ++rr) rowptr[rr] = (int32_t)nnz;
  colidx[p] = (int32_t)cols[p];
  vals[2 * p] = vx[p];
  vals[2 * p + 1] = vy ? vy[p] : 0.f;
}

// out[v][c][0..1] = (gradX @ x, gradY @ x)  -- the reference's (V,C,2) layout, layers.py:216-223
__global__ void grad_spmm_pair_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                                      const float2* __restrict__ vals, const float* __restrict__ x, int64_t V,
                                      int C, float* __restrict__ out) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= V) return;
  const int s = rowptr[row], e = rowptr[row + 1];
  for (int c = lane; c < C; c += 32) {
    float gx = 0.f, gy = 0.f;
    for (int p = s; p < e; ++p) {
      const float2 g = __ldg(vals + p);
      const float xv = __ldg(x + (int64_t)__ldg(colidx + p) * C + c);
      gx = fmaf(g.x, xv, gx);
      gy = fmaf(g.y, xv, gy);
    }
    reinterpret_cast<float2*>(out)[row * C + c] = make_float2(gx, gy);
  }
}

struct Acc4 {
  float4 gX, gY, bre, bim;
};

// tanh(x) = 1 - 2 / (exp(2x) + 1) with the hardware exp2 and fast division: ~6 instructions instead of tanhf's ~30
// (the gather kernel issues instructions on 53 % of its cycles, profiles/r01: the four tanhf per lane were a fifth of
// them).  Absolute error <= ~1.5e-7 over the whole range (saturates to +-1, NaN propagates); every gather variant
// uses this one function so that they stay bit-identical to each other.
__device__ __forceinline__ float feat_tanh(float x) { return dn_feat_tanh(x); }

template <bool ROT>
__device__ __forceinline__ Acc4 gather_row(const int32_t* __restrict__ colidx, const float2* __restrict__ vals,
                                           const float* __restrict__ xd, const float* __restrict__ pq, int ld_pq,
                                           int C, int s, int e, int c4) {
  Acc4 a;
  a.gX = a.gY = a.bre = a.bim = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
  for (int p = s; p < e; ++p) {
    const int64_t col = __ldg(colidx + p);
    const float2 g = __ldg(vals + p);
    const float4 x = ldg4(xd + col * C + c4 * 4);
    const float4 P = ldg4(pq + col * ld_pq + c4 * 4);
    a.gX.x = fmaf(g.x, x.x, a.gX.x); a.gX.y = fmaf(g.x, x.y, a.gX.y);
    a.gX.z = fmaf(g.x, x.z, a.gX.z); a.gX.w = fmaf(g.x, x.w, a.gX.w);
    a.gY.x = fmaf(g.y, x.x, a.gY.x); a.gY.y = fmaf(g.y, x.y, a.gY.y);
    a.gY.z = fmaf(g.y, x.z, a.gY.z); a.gY.w = fmaf(g.y, x.w, a.gY.w);
    a.bre.x = fmaf(g.x, P.x, a.bre.x); a.bre.y = fmaf(g.x, P.y, a.bre.y);
    a.bre.z = fmaf(g.x, P.z, a.bre.z); a.bre.w = fmaf(g.x, P.w, a.bre.w);
    a.bim.x = fmaf(g.y, P.x, a.bim.x); a.bim.y = fmaf(g.y, P.y, a.bim.y);
    a.bim.z = fmaf(g.y, P.z, a.bim.z); a.bim.w = fmaf(g.y, P.w, a.bim.w);
    if (ROT) {
      const float4 Q = ldg4(pq + col * ld_pq + C + c4 * 4);
      a.bre.x = fmaf(-g.y, Q.x, a.bre.x); a.bre.y = fmaf(-g.y, Q.y, a.bre.y);
      a.bre.z = fmaf(-g.y, Q.z, a.bre.z); a.bre.w = fmaf(-g.y, Q.w, a.bre.w);
      a.bim.x = fmaf(g.x, Q.x, a.bim.x); a.bim.y = fmaf(g.x, Q.y, a.bim.y);
      a.bim.z = fmaf(g.x, Q.z, a.bim.z); a.bim.w = fmaf(g.x, Q.w, a.bim.w);
    }
  }
  return a;
}

// feat = tanh(gX*Bre + gY*Bim), Bre/Bim gathered from P = xd A_re^T, Q = xd A_im^T (layers.py:121-130)
template <bool ROT>
__global__ void __launch_bounds__(256) spmm_features_kernel(const int32_t* __restrict__ rowptr,
                                                            const int32_t* __restrict__ colidx,
                                                            const float2* __restrict__ vals,
                                                            const float* __restrict__ xd, const float* __restrict__ pq,
                                                            int ld_pq, int64_t V, int C, int G,
                                                            float* __restrict__ feat) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t row = warp * (32 / G) + lane / G;
  const int gl = lane % G;
  if (row >= V) return;
  const int s = __ldg(rowptr + row), e = __ldg(rowptr + row + 1);
  for (int c4 = gl; c4 < (C >> 2); c4 += G) {
    const Acc4 a = gather_row<ROT>(colidx, vals, xd, pq, ld_pq, C, s, e, c4);
    float4 o;
    o.x = feat_tanh(fmaf(a.gX.x, a.bre.x, a.gY.x * a.bim.x));
    o.y = feat_tanh(fmaf(a.gX.y, a.bre.y, a.gY.y * a.bim.y));
    o.z = feat_tanh(fmaf(a.gX.z, a.bre.z, a.gY.z * a.bim.z));
    o.w = feat_tanh(fmaf(a.gX.w, a.bre.w, a.gY.w * a.bim.w));
    *reinterpret_cast<float4*>(feat + row * C + c4 * 4) = o;
  }
}

__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
// d = a * b + d on both fp32 halves (sm_100 FFMA2)
__device__ __forceinline__ void fma2(unsigned long long& d, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}

// ---------------------------------------------------------------------------------------------
// Block gather (C a multiple of 128): one CTA per 64 consecutive rows.
//   * the block's CSR metadata (rowptr slice, every (col, gx, gy) triple) is staged in shared memory by ONE coalesced
//     pass: the per-row dependent chain rowptr -> colidx -> neighbour rows (three DRAM/L2 latencies in the warp-per-row
//     kernel) becomes one latency per 64 rows plus the gathers themselves;
//   * a warp issues every neighbour-row load of a batch of NB entries (3 x NB independent 16-byte loads per lane)
//     before the first FMA; 8 warps walk 8 consecutive rows at a time, so the band structure of a locally ordered
//     mesh hits L1;
//   * packed fp32x2 FMAs (fma.rn.f32x2: two IEEE fp32 FMAs per instruction, bit-identical to fmaf).
// Entry order = CSR order and the arithmetic per element is the same fmaf sequence as gather_row: bit-identical output.
// ---------------------------------------------------------------------------------------------
constexpr int GB_ROWS = 64;      // rows per CTA
constexpr int GB_NNZ = 1024;     // staged entries per CTA (entries past it are read from global memory)

struct __align__(16) GxyEnt { int col; int pad; float gx, gy; };   // (gx, gy) 8-byte aligned: one LDS.64

// one CSR entry of the (x, P, Q) gather: three 16-byte slices of the neighbour's rows, then 12 FFMA2
#define DN_FEAT_LOAD(J, ENT)                                                                         \
  const char* pr##J;                                                                                 \
  ulonglong2 x##J, P##J, Q##J = make_ulonglong2(0ull, 0ull);                                         \
  {                                                                                                  \
    const int64_t col = (ENT).col;                                                                   \
    x##J = __ldg(reinterpret_cast<const ulonglong2*>(xb + col * x_row_bytes));                       \
    pr##J = pb + col * pq_row_bytes;                                                                 \
    P##J = __ldg(reinterpret_cast<const ulonglong2*>(pr##J));                                        \
    if (ROT) Q##J = __ldg(reinterpret_cast<const ulonglong2*>(pr##J + x_row_bytes));                 \
  }
// (the weights are re-read from the staged entry at FMA time: a broadcast LDS.64 is cheaper than 14 live registers)
#define DN_FEAT_FMA(J, ENT)                                                                          \
  {                                                                                                  \
    const float2 w = *reinterpret_cast<const float2*>(&(ENT).gx);                                    \
    const unsigned long long gx2 = pack2(w.x, w.x), gy2 = pack2(w.y, w.y);                           \
    fma2(gX0, gx2, x##J.x); fma2(gX1, gx2, x##J.y);                                                  \
    fma2(gY0, gy2, x##J.x); fma2(gY1, gy2, x##J.y);                                                  \
    fma2(re0, gx2, P##J.x); fma2(re1, gx2, P##J.y);                                                  \
    fma2(im0, gy2, P##J.x); fma2(im1, gy2, P##J.y);                                                  \
    if (ROT) {                                                                                       \
      const unsigned long long ngy2 = pack2(-w.y, -w.y);                                             \
      fma2(re0, ngy2, Q##J.x); fma2(re1, ngy2, Q##J.y);                                              \
      fma2(im0, gx2, Q##J.x); fma2(im1, gx2, Q##J.y);                                                \
    }                                                                                                \
  }

// (Same staging as spmm_gxy_blk_kernel below: 16-byte entry records, unpredicated full batches -- the first version,
// with per-entry predicates and separate col / value arrays, spent half of its issue slots on bookkeeping.)
template <bool ROT, int NH>
__global__ void __launch_bounds__(256, 2)
spmm_features_blk_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                         const float2* __restrict__ vals, const float* __restrict__ xd,
                         const float* __restrict__ pq, int ld_pq, int64_t V, float* __restrict__ feat) {
  constexpr int C = 128 * NH;          // a warp covers 128 channels per pass (one float4 per lane), NH passes per row
  constexpr int64_t x_row_bytes = (int64_t)C * 4;
  __shared__ int s_rp[GB_ROWS + 1];
  __shared__ GxyEnt s_e[GB_NNZ];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * GB_ROWS;
  const int nrows = (int)((V - base) < GB_ROWS ? (V - base) : GB_ROWS);
  if ((int)threadIdx.x <= nrows) s_rp[threadIdx.x] = __ldg(rowptr + base + threadIdx.x);
  __syncthreads();
  const int e0 = s_rp[0];
  const int tot = s_rp[nrows] - e0;
  const bool staged = tot <= GB_NNZ;                              // (block-uniform)
  if (staged) {
    for (int i = threadIdx.x; i < tot; i += 256) {
      const float2 g = __ldg(vals + e0 + i);
      GxyEnt en;
      en.col = __ldg(colidx + e0 + i); en.gx = g.x; en.gy = g.y; en.pad = 0;
      s_e[i] = en;
    }
  }
  __syncthreads();
  const int64_t pq_row_bytes = (int64_t)ld_pq * 4;
#pragma unroll 1
  for (int rh = warp; rh < nrows * NH; rh += 8) {
    const int r = rh / NH, h = rh % NH;
    const char* xb = reinterpret_cast<const char*>(xd) + h * 512 + lane * 16;
    const char* pb = reinterpret_cast<const char*>(pq) + h * 512 + lane * 16;
    const int s = s_rp[r] - e0, e = s_rp[r + 1] - e0;
    unsigned long long gX0 = 0ull, gX1 = 0ull, gY0 = 0ull, gY1 = 0ull, re0 = 0ull, re1 = 0ull, im0 = 0ull, im1 = 0ull;
    if (staged) {
      int p = s;
#pragma unroll 1
      for (; p + 7 <= e; p += 7) {                                // full batches: 21 independent loads, no predicates
        DN_FEAT_LOAD(0, s_e[p]) DN_FEAT_LOAD(1, s_e[p + 1]) DN_FEAT_LOAD(2, s_e[p + 2]) DN_FEAT_LOAD(3, s_e[p + 3])
        DN_FEAT_LOAD(4, s_e[p + 4]) DN_FEAT_LOAD(5, s_e[p + 5]) DN_FEAT_LOAD(6, s_e[p + 6])
        DN_FEAT_FMA(0, s_e[p]) DN_FEAT_FMA(1, s_e[p + 1]) DN_FEAT_FMA(2, s_e[p + 2]) DN_FEAT_FMA(3, s_e[p + 3])
        DN_FEAT_FMA(4, s_e[p + 4]) DN_FEAT_FMA(5, s_e[p + 5]) DN_FEAT_FMA(6, s_e[p + 6])
      }
#pragma unroll 1
      for (; p + 2 <= e; p += 2) {                                // remainder: pairs, then a single entry
        DN_FEAT_LOAD(0, s_e[p]) DN_FEAT_LOAD(1, s_e[p + 1])
        DN_FEAT_FMA(0, s_e[p]) DN_FEAT_FMA(1, s_e[p + 1])
      }
      if (p < e) {
        DN_FEAT_LOAD(0, s_e[p])
        DN_FEAT_FMA(0, s_e[p])
      }
    } else {
#pragma unroll 1
      for (int p = s; p < e; ++p) {                               // (a block with more than GB_NNZ entries)
        GxyEnt en;
        const float2 g = __ldg(vals + e0 + p);
        en.col = __ldg(colidx + e0 + p); en.gx = g.x; en.gy = g.y; en.pad = 0;
        DN_FEAT_LOAD(0, en)
        DN_FEAT_FMA(0, en)
      }
    }
    float gXv[4], gYv[4], rev[4], imv[4];
    unpack2(gX0, gXv[0], gXv[1]); unpack2(gX1, gXv[2], gXv[3]);
    unpack2(gY0, gYv[0], gYv[1]); unpack2(gY1, gYv[2], gYv[3]);
    unpack2(re0, rev[0], rev[1]); unpack2(re1, rev[2], rev[3]);
    unpack2(im0, imv[0], imv[1]); unpack2(im1, imv[2], imv[3]);
    float4 o;
    o.x = feat_tanh(fmaf(gXv[0], rev[0], gYv[0] * imv[0]));
    o.y = feat_tanh(fmaf(gXv[1], rev[1], gYv[1] * imv[1]));
    o.z = feat_tanh(fmaf(gXv[2], rev[2], gYv[2] * imv[2]));
    o.w = feat_tanh(fmaf(gXv[3], rev[3], gYv[3] * imv[3]));
    *reinterpret_cast<float4*>(feat + (base + r) * C + h * 128 + lane * 4) = o;
  }
}
#undef DN_FEAT_LOAD
#undef DN_FEAT_FMA

// The same block gather for the tensor-core gradient-features route: only x_diffuse is gathered (7 x 512 B per
// vertex instead of 7 x 1.5 KB) and the raw tangent gradients are written out,
//     gxy[v] = [ sum_j gx_vj x_j | sum_j gy_vj x_j ]                                       (layers.py:216-223)
// the complex-linear map, the inner product and the tanh follow as a tcgen05 GEMM with a fused epilogue (rows_chain3,
// has_res == 3).  Entry order = CSR order, fmaf per element (as FFMA2).


// One CSR entry of the x-only gather: the neighbour row's 16-byte slice is loaded, then 4 FFMA2 -- gX += gx * x, gY += gy * x
#define DN_GXY_LOAD(J, ENT)                                                                          \
  const int4 en##J = *reinterpret_cast<const int4*>(&(ENT));                                         \
  const ulonglong2 x##J = __ldg(reinterpret_cast<const ulonglong2*>(xb + (int64_t)en##J.x * x_row_bytes));
#define DN_GXY_FMA(J)                                                                                \
  {                                                                                                  \
    const float wx = __int_as_float(en##J.z), wy = __int_as_float(en##J.w);                          \
    const unsigned long long gx2 = pack2(wx, wx), gy2 = pack2(wy, wy);                               \
    fma2(gX0, gx2, x##J.x); fma2(gX1, gx2, x##J.y);                                                  \
    fma2(gY0, gy2, x##J.x); fma2(gY1, gy2, x##J.y);                                                  \
  }

// The instruction count is what bounds this kernel (ncu: 71 % issue-active in the first version, whose per-entry
// predicates and two staging arrays cost ~4x the useful instructions): entries are staged as 16-byte records (one
// broadcast LDS.128 per entry), full batches of 7 run without predicates, and blocks whose entries do not fit the
// staging buffer take a separate (generic) path.
template <int NH>
__global__ void __launch_bounds__(256, 3)
spmm_gxy_blk_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                    const float2* __restrict__ vals, const float* __restrict__ xd, int64_t V, float* __restrict__ gxy) {
  constexpr int C = 128 * NH;
  constexpr int64_t x_row_bytes = (int64_t)C * 4;
  __shared__ int s_rp[GB_ROWS + 1];
  __shared__ GxyEnt s_e[GB_NNZ];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t base = (int64_t)blockIdx.x * GB_ROWS;
  const int nrows = (int)((V - base) < GB_ROWS ? (V - base) : GB_ROWS);
  if ((int)threadIdx.x <= nrows) s_rp[threadIdx.x] = __ldg(rowptr + base + threadIdx.x);
  __syncthreads();
  const int e0 = s_rp[0];
  const int tot = s_rp[nrows] - e0;
  const bool staged = tot <= GB_NNZ;                              // (block-uniform)
  if (staged) {
    for (int i = threadIdx.x; i < tot; i += 256) {
      const float2 g = __ldg(vals + e0 + i);
      GxyEnt en;
      en.col = __ldg(colidx + e0 + i); en.gx = g.x; en.gy = g.y; en.pad = 0;
      s_e[i] = en;
    }
  }
  __syncthreads();
#pragma unroll 1
  for (int rh = warp; rh < nrows * NH; rh += 8) {
    const int r = rh / NH, h = rh % NH;
    const char* xb = reinterpret_cast<const char*>(xd) + h * 512 + lane * 16;
    const int s = s_rp[r] - e0, e = s_rp[r + 1] - e0;
    unsigned long long gX0 = 0ull, gX1 = 0ull, gY0 = 0ull, gY1 = 0ull;
    if (staged) {
      int p = s;
#pragma unroll 1
      for (; p + 7 <= e; p += 7) {                                // full batches: seven independent loads, no predicates
        DN_GXY_LOAD(0, s_e[p]) DN_GXY_LOAD(1, s_e[p + 1]) DN_GXY_LOAD(2, s_e[p + 2]) DN_GXY_LOAD(3, s_e[p + 3])
        DN_GXY_LOAD(4, s_e[p + 4]) DN_GXY_LOAD(5, s_e[p + 5]) DN_GXY_LOAD(6, s_e[p + 6])
        DN_GXY_FMA(0) DN_GXY_FMA(1) DN_GXY_FMA(2) DN_GXY_FMA(3) DN_GXY_FMA(4) DN_GXY_FMA(5) DN_GXY_FMA(6)
      }
#pragma unroll 1
      for (; p + 2 <= e; p += 2) {                                // remainder: pairs, then a single entry
        DN_GXY_LOAD(0, s_e[p]) DN_GXY_LOAD(1, s_e[p + 1])
        DN_GXY_FMA(0) DN_GXY_FMA(1)
      }
      if (p < e) {
        DN_GXY_LOAD(0, s_e[p])
        DN_GXY_FMA(0)
      }
    } else {
#pragma unroll 1
      for (int p = s; p < e; ++p) {                               // (a block with more than GB_NNZ entries)
        GxyEnt en;
        const float2 g = __ldg(vals + e0 + p);
        en.col = __ldg(colidx + e0 + p); en.gx = g.x; en.gy = g.y; en.pad = 0;
        DN_GXY_LOAD(0, en)
        DN_GXY_FMA(0)
      }
    }
    char* o = reinterpret_cast<char*>(gxy + (base + r) * (2 * C)) + h * 512 + lane * 16;
    *reinterpret_cast<ulonglong2*>(o) = make_ulonglong2(gX0, gX1);
    *reinterpret_cast<ulonglong2*>(o + x_row_bytes) = make_ulonglong2(gY0, gY1);
  }
}
#undef DN_GXY_LOAD
#undef DN_GXY_FMA

// Patch variant (dn_patches, built once for resident operators): one CTA per patch of graph-adjacent rows.
// Phase 1 copies the patch's distinct neighbour rows of x_diffuse and [P|Q] into shared memory, coalesced, each row
// exactly once; phase 2 is the same gather as above but out of shared memory.  At V = 200k the plain kernel moves
// ~1.1 GB from L2 into the SMs (every neighbour row is re-fetched by ~half of the vertices that touch it: 47 % L1
// hits); here it is (distinct rows / rows) x 1.5 KB per vertex.  Entries keep their CSR order and the arithmetic is
// gather_row's, so the result is bit-identical.
template <bool ROT>
__global__ void __launch_bounds__(512) spmm_features_patch_kernel(const dn_patches P, const float* __restrict__ xd,
                                                                  const float* __restrict__ pq, int ld_pq, int C,
                                                                  float* __restrict__ feat) {
  extern __shared__ float4 sm4[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int xq = C >> 2, pqq = ld_pq >> 2, rowf4 = xq + pqq;
  const int p = blockIdx.x;
  const int s0 = __ldg(P.src_ptr + p), ns = __ldg(P.src_ptr + p + 1) - s0;
  const int t0 = __ldg(P.tgt_ptr + p), nt = __ldg(P.tgt_ptr + p + 1) - t0;
  const float2* vals = reinterpret_cast<const float2*>(P.vals);

  // per-row metadata of this warp's target, one entry per lane (coalesced), fetched one round ahead so that its
  // latency hides behind the row copies (round 0) or the previous round's arithmetic
  struct Meta { int64_t row; int es, n; int lc; float2 g; };
  auto load_meta = [&](int i) {
    Meta m;
    m.row = 0; m.es = 0; m.n = 0; m.lc = 0; m.g = make_float2(0.f, 0.f);
    if (i < nt) {
      m.row = __ldg(P.tgt + t0 + i);
      m.es = __ldg(P.ent_ptr + t0 + i);
      m.n = __ldg(P.ent_ptr + t0 + i + 1) - m.es;
      if (lane < m.n) { m.lc = __ldg(P.lcol + m.es + lane); m.g = __ldg(vals + m.es + lane); }
    }
    return m;
  };
  Meta cur = load_meta(warp);

  // phase 1: distinct neighbour rows -> shared memory, four rows (12 x 16 B at C = 128) in flight per lane
  for (int r = warp; r < ns; r += 4 * nwarps) {
    int64_t row[4];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ok[u] = r + u * nwarps < ns;
      row[u] = __ldg(P.src_rows + s0 + (ok[u] ? r + u * nwarps : r));
    }
    for (int c4 = lane; c4 < xq; c4 += 32) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ldg4(xd + row[u] * C + 4 * c4);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u]) sm4[(size_t)(r + u * nwarps) * rowf4 + c4] = v[u];
    }
    for (int c4 = lane; c4 < pqq; c4 += 32) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ldg4(pq + row[u] * ld_pq + 4 * c4);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u]) sm4[(size_t)(r + u * nwarps) * rowf4 + xq + c4] = v[u];
    }
  }
  __syncthreads();

  // phase 2: the gather, out of shared memory; entries in CSR order, gather_row's arithmetic
  for (int i = warp; i < nt; i += nwarps) {
    const Meta nxt = load_meta(i + nwarps);
    for (int c4 = lane; c4 < xq; c4 += 32) {
      Acc4 a;
      a.gX = a.gY = a.bre = a.bim = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int base = 0; base < cur.n; base += 32) {
        int lc_l = cur.lc;
        float2 g_l = cur.g;
        if (base > 0) {                                            // rows longer than a warp: next 32 entries
          lc_l = 0; g_l = make_float2(0.f, 0.f);
          if (base + lane < cur.n) { lc_l = __ldg(P.lcol + cur.es + base + lane); g_l = __ldg(vals + cur.es + base + lane); }
        }
        const int cnt = (cur.n - base) < 32 ? (cur.n - base) : 32;
        for (int e = 0; e < cnt; ++e) {
          const int lc = __shfl_sync(0xffffffffu, lc_l, e);
          float2 g;
          g.x = __shfl_sync(0xffffffffu, g_l.x, e);
          g.y = __shfl_sync(0xffffffffu, g_l.y, e);
          const float4* src = sm4 + (size_t)lc * rowf4;
          const float4 x = src[c4];
          const float4 Pv = src[xq + c4];
          a.gX.x = fmaf(g.x, x.x, a.gX.x); a.gX.y = fmaf(g.x, x.y, a.gX.y);
          a.gX.z = fmaf(g.x, x.z, a.gX.z); a.gX.w = fmaf(g.x, x.w, a.gX.w);
          a.gY.x = fmaf(g.y, x.x, a.gY.x); a.gY.y = fmaf(g.y, x.y, a.gY.y);
          a.gY.z = fmaf(g.y, x.z, a.gY.z); a.gY.w = fmaf(g.y, x.w, a.gY.w);
          a.bre.x = fmaf(g.x, Pv.x, a.bre.x); a.bre.y = fmaf(g.x, Pv.y, a.bre.y);
          a.bre.z = fmaf(g.x, Pv.z, a.bre.z); a.bre.w = fmaf(g.x, Pv.w, a.bre.w);
          a.bim.x = fmaf(g.y, Pv.x, a.bim.x); a.bim.y = fmaf(g.y, Pv.y, a.bim.y);
          a.bim.z = fmaf(g.y, Pv.z, a.bim.z); a.bim.w = fmaf(g.y, Pv.w, a.bim.w);
          if (ROT) {
            const float4 Q = src[2 * xq + c4];
            a.bre.x = fmaf(-g.y, Q.x, a.bre.x); a.bre.y = fmaf(-g.y, Q.y, a.bre.y);
            a.bre.z = fmaf(-g.y, Q.z, a.bre.z); a.bre.w = fmaf(-g.y, Q.w, a.bre.w);
            a.bim.x = fmaf(g.x, Q.x, a.bim.x); a.bim.y = fmaf(g.x, Q.y, a.bim.y);
            a.bim.z = fmaf(g.x, Q.z, a.bim.z); a.bim.w = fmaf(g.x, Q.w, a.bim.w);
          }
        }
      }
      float4 o;
      o.x = feat_tanh(fmaf(a.gX.x, a.bre.x, a.gY.x * a.bim.x));
      o.y = feat_tanh(fmaf(a.gX.y, a.bre.y, a.gY.y * a.bim.y));
      o.z = feat_tanh(fmaf(a.gX.z, a.bre.z, a.gY.z * a.bim.z));
      o.w = feat_tanh(fmaf(a.gX.w, a.bre.w, a.gY.w * a.bim.w));
      *reinterpret_cast<float4*>(feat + cur.row * C + c4 * 4) = o;
    }
    cur = nxt;
  }
}

// U[v] = [dd*Bre | dd*Bim | dd*gX | dd*gY],  dd = dfeat * (1 - feat^2)
template <bool ROT>
__global__ void __launch_bounds__(256) features_bwd_local_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float2* __restrict__ vals,
    const float* __restrict__ xd, const float* __restrict__ pq, int ld_pq, const float* __restrict__ feat,
    const float* __restrict__ dfeat, int64_t V, int C, int G, float* __restrict__ U) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t row = warp * (32 / G) + lane / G;
  const int gl = lane % G;
  if (row >= V) return;
  const int s = __ldg(rowptr + row), e = __ldg(rowptr + row + 1);
  for (int c4 = gl; c4 < (C >> 2); c4 += G) {
    const Acc4 a = gather_row<ROT>(colidx, vals, xd, pq, ld_pq, C, s, e, c4);
    const float4 f = ldg4(feat + row * C + c4 * 4);
    const float4 d = ldg4(dfeat + row * C + c4 * 4);
    float4 dd;
    dd.x = d.x * (1.f - f.x * f.x); dd.y = d.y * (1.f - f.y * f.y);
    dd.z = d.z * (1.f - f.z * f.z); dd.w = d.w * (1.f - f.w * f.w);
    float* u = U + row * 4 * C + c4 * 4;
    *reinterpret_cast<float4*>(u) = make_float4(dd.x * a.bre.x, dd.y * a.bre.y, dd.z * a.bre.z, dd.w * a.bre.w);
    *reinterpret_cast<float4*>(u + C) = make_float4(dd.x * a.bim.x, dd.y * a.bim.y, dd.z * a.bim.z, dd.w * a.bim.w);
    *reinterpret_cast<float4*>(u + 2 * C) = make_float4(dd.x * a.gX.x, dd.y * a.gX.y, dd.z * a.gX.z, dd.w * a.gX.w);
    *reinterpret_cast<float4*>(u + 3 * C) = make_float4(dd.x * a.gY.x, dd.y * a.gY.y, dd.z * a.gY.z, dd.w * a.gY.w);
  }
}

// transpose gather over the CSR of G^T:  dxd = GX^T U1 + GY^T U2;  dP = GX^T U3 + GY^T U4;
// dQ = -GY^T U3 + GX^T U4
template <bool ROT>
__global__ void __launch_bounds__(256) features_bwd_transpose_kernel(
    const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx, const float2* __restrict__ vals,
    const float* __restrict__ U, int64_t V, int C, int G, float* __restrict__ dxd, float* __restrict__ dP,
    float* __restrict__ dQ, int64_t ld_pq) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t row = warp * (32 / G) + lane / G;
  const int gl = lane % G;
  if (row >= V) return;
  const int s = __ldg(rowptr + row), e = __ldg(rowptr + row + 1);
  for (int c4 = gl; c4 < (C >> 2); c4 += G) {
    float4 ax = make_float4(0.f, 0.f, 0.f, 0.f), ap = ax, aq = ax;
    for (int p = s; p < e; ++p) {
      const int64_t i = __ldg(colidx + p);
      const float2 g = __ldg(vals + p);
      const float* u = U + i * 4 * C + c4 * 4;
      const float4 u1 = ldg4(u), u2 = ldg4(u + C), u3 = ldg4(u + 2 * C), u4 = ldg4(u + 3 * C);
      ax.x += g.x * u1.x + g.y * u2.x; ax.y += g.x * u1.y + g.y * u2.y;
      ax.z += g.x * u1.z + g.y * u2.z; ax.w += g.x * u1.w + g.y * u2.w;
      ap.x += g.x * u3.x + g.y * u4.x; ap.y += g.x * u3.y + g.y * u4.y;
      ap.z += g.x * u3.z + g.y * u4.z; ap.w += g.x * u3.w + g.y * u4.w;
      if (ROT) {
        aq.x += g.x * u4.x - g.y * u3.x; aq.y += g.x * u4.y - g.y * u3.y;
        aq.z += g.x * u4.z - g.y * u3.z; aq.w += g.x * u4.w - g.y * u3.w;
      }
    }
    *reinterpret_cast<float4*>(dxd + row * C + c4 * 4) = ax;
    *reinterpret_cast<float4*>(dP + row * ld_pq + c4 * 4) = ap;
    if (ROT) *reinterpret_cast<float4*>(dQ + row * ld_pq + c4 * 4) = aq;
  }
}

__global__ void deinterleave_vc2_kernel(const float2* __restrict__ vc2, int64_t V, int C, float* __restrict__ g01) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= V * C) return;
  const int64_t v = idx / C;
  const int c = (int)(idx % C);
  const float2 g = __ldg(vc2 + idx);
  g01[v * 2 * C + c] = g.x;
  g01[v * 2 * C + C + c] = g.y;
}

__global__ void complex_dots_tanh_kernel(const float* __restrict__ g01, const float* __restrict__ b01, int64_t V,
                                         int C, float* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= V * C) return;
  const int64_t v = idx / C;
  const int c = (int)(idx % C);
  const float d = g01[v * 2 * C + c] * b01[v * 2 * C + c] + g01[v * 2 * C + C + c] * b01[v * 2 * C + C + c];
  out[idx] = tanhf(d);
}

inline int pick_group(int C) {
  int g = 1;
  while (g * 2 <= 32 && g * 2 <= (C >> 2)) g *= 2;
  return g;
}

}  // namespace

// =============================================================================================
// host launchers
// =============================================================================================
int simt_rows_gemm(const DnRowsSrc& src, const DnLayer& L, int64_t V, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (!L.out) return DN_ERR_INVALID_ARGUMENT;
  bool vec = true;
  int ktot = 0;
  for (int i = 0; i < src.nsrc; ++i) {
    vec = vec && (src.width[i] % 4 == 0) && (src.ld[i] % 4 == 0) &&
          ((reinterpret_cast<uintptr_t>(src.ptr[i]) & 15) == 0);
    ktot += src.width[i];
  }
  if (ktot != L.K) return DN_ERR_INVALID_ARGUMENT;
  vec = vec && (L.ldw % 4 == 0) && ((reinterpret_cast<uintptr_t>(L.W) & 15) == 0) &&
        (!L.W2 || (reinterpret_cast<uintptr_t>(L.W2) & 15) == 0);
  dim3 grid((unsigned)((V + RG_BM - 1) / RG_BM), (unsigned)((L.N + RG_BN - 1) / RG_BN));
  if (vec)
    rows_gemm_kernel<true><<<grid, 256, 0, st>>>(src, L, V);
  else
    rows_gemm_kernel<false><<<grid, 256, 0, st>>>(src, L, V);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int simt_atb_partial_st(const float* A, int64_t lda, int I, const float* B, int64_t ldb, int J, const float* scale,
                        int64_t V, float* ws, int64_t ws_floats, int* P_out, cudaStream_t st) {
  const int tiles = ((I + 63) / 64) * ((J + 63) / 64);
  int P = (int)((V + 2047) / 2048);
  const int maxP = (4 * 148) / tiles > 1 ? (4 * 148) / tiles : 1;
  if (P > maxP) P = maxP;
  if (P < 1) P = 1;
  while ((int64_t)P * I * J > ws_floats && P > 1) --P;
  if ((int64_t)P * I * J > ws_floats) return DN_ERR_WORKSPACE;
  int64_t rps = (V + P - 1) / P;
  rps = (rps + 15) / 16 * 16;
  if (rps < 16) rps = 16;
  P = (int)((V + rps - 1) / rps);
  if (P < 1) P = 1;
  atb_partial_kernel<<<dim3(tiles, P), 256, 0, st>>>(A, lda, I, B, ldb, J, scale, V, rps, ws);
  DN_LAUNCH_CHECK();
  *P_out = P;
  return DN_OK;
}

int simt_atb(const float* A, int64_t lda, int I, const float* B, int64_t ldb, int J, const float* scale, int64_t V,
             float* out, int64_t ld_out, int accumulate, float* ws, int64_t ws_floats, cudaStream_t st) {
  int P = 0;
  int rc = simt_atb_partial_st(A, lda, I, B, ldb, J, scale, V, ws, ws_floats, &P, st);
  if (rc) return rc;
  const int64_t n = (int64_t)I * J;
  reduce_partials_ld_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ws, P, I, J, out, ld_out, accumulate);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int simt_colsum(const float* A, int64_t lda, int N, int64_t V, float* out, int accumulate, cudaStream_t st) {
  if (!accumulate) DN_CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(float) * N, st));
  if (V <= 0) return DN_OK;
  dim3 grid((unsigned)((V + 255) / 256), (unsigned)((N + 31) / 32));
  colsum_kernel<<<grid, dim3(32, 8), 0, st>>>(A, lda, N, V, out);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_spectral_scale(const float* partial, int P, const float* evals, float* time, int K, int C,
                          float* x_spec_out, float* S_out, int clamp_writeback, cudaStream_t st) {
  spectral_scale_kernel<<<(K * C + 63) / 64, 256, 0, st>>>(partial, P, evals, time, K, C, x_spec_out, S_out,
                                                            clamp_writeback);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_reduce_partials(const float* partial, int P, int64_t n, float* out, cudaStream_t st) {
  reduce_partials_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partial, P, n, out);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_reduce_partials_ld(const float* partial, int P, int rows, int cols, float* out, int64_t ld_out,
                              int accumulate, cudaStream_t st) {
  reduce_partials_ld_kernel<<<(unsigned)((rows * cols + 255) / 256), 256, 0, st>>>(partial, P, rows, cols, out, ld_out,
                                                                                   accumulate);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_spectral_bwd(const float* gs_partial, int P, const float* evals, const float* time, const float* x_spec,
                        int K, int C, float* dS, float* grad_time, cudaStream_t st) {
  spectral_bwd_kernel<<<(C + 63) / 64, 64, 0, st>>>(gs_partial, P, evals, time, x_spec, K, C, dS, grad_time);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_csr_from_coo(const int64_t* rows, const int64_t* cols, const float* vx, const float* vy, int64_t nnz,
                        int64_t V, int32_t* rowptr, int32_t* colidx, float* vals, cudaStream_t st) {
  if (nnz == 0) {
    DN_CUDA_TRY(cudaMemsetAsync(rowptr, 0, sizeof(int32_t) * (V + 1), st));
    return DN_OK;
  }
  csr_from_coo_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(rows, cols, vx, vy, nnz, V, rowptr, colidx, vals);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_grad_spmm_pair(const dn_csr* g, const float* x, int64_t V, int C, float* out, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  const int64_t threads = V * 32;
  grad_spmm_pair_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(
      g->rowptr, g->colidx, reinterpret_cast<const float2*>(g->vals), x, V, C, out);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_spmm_features(const dn_csr* g, const float* xd, const float* pq, int rotations, int64_t V, int C,
                         float* feat, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (C % 4) return DN_ERR_UNSUPPORTED;
  // C == 128 only: that is the shape validated on the GPU (bit-identical to the plain kernel, both ROT variants); the
  // phase-2 shuffles also assume every lane owns a float4 of the row (C/4 a multiple of 32)
  if (g->patches && g->patches->n_patches > 0 && C == 128) {
    const dn_patches& P = *g->patches;
    const int ld = rotations ? 2 * C : C;
    const size_t smem = (size_t)P.max_src * (size_t)(C + ld) * 4;
    if (smem <= 227 * 1024) {
      static size_t attr_set[2] = {0, 0};
      if (smem > attr_set[rotations ? 1 : 0]) {
        DN_CUDA_TRY(rotations ? cudaFuncSetAttribute(spmm_features_patch_kernel<true>,
                                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(spmm_features_patch_kernel<false>,
                                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[rotations ? 1 : 0] = smem;
      }
      if (rotations) spmm_features_patch_kernel<true><<<(unsigned)P.n_patches, 512, smem, st>>>(P, xd, pq, ld, C, feat);
      else spmm_features_patch_kernel<false><<<(unsigned)P.n_patches, 512, smem, st>>>(P, xd, pq, ld, C, feat);
      DN_LAUNCH_CHECK();
      return DN_OK;
    }
  }
  const float2* vals = reinterpret_cast<const float2*>(g->vals);
  // block gather at C = 128 / 256: measured (profiles/r02_ab_gather_blk.log, V=200k) 175 us (281 permuted) vs 181 (347)
  // for the warp-per-row kernel below, which serves the other widths
  if (C == 128 || C == 256) {
    const unsigned ctas = (unsigned)((V + GB_ROWS - 1) / GB_ROWS);
    const int ld = rotations ? 2 * C : C;
#define DN_BLK_LAUNCH(ROT_, NH_) \
    spmm_features_blk_kernel<ROT_, NH_><<<ctas, 256, 0, st>>>(g->rowptr, g->colidx, vals, xd, pq, ld, V, feat)
    if (rotations) { if (C == 128) DN_BLK_LAUNCH(true, 1); else DN_BLK_LAUNCH(true, 2); }
    else { if (C == 128) DN_BLK_LAUNCH(false, 1); else DN_BLK_LAUNCH(false, 2); }
#undef DN_BLK_LAUNCH
    DN_LAUNCH_CHECK();
    return DN_OK;
  }
  const int G = pick_group(C);
  const int64_t warps = (V + (32 / G) - 1) / (32 / G);
  const unsigned blocks = (unsigned)((warps * 32 + 255) / 256);
  if (rotations)
    spmm_features_kernel<true><<<blocks, 256, 0, st>>>(g->rowptr, g->colidx, vals, xd, pq, 2 * C, V, C, G, feat);
  else
    spmm_features_kernel<false><<<blocks, 256, 0, st>>>(g->rowptr, g->colidx, vals, xd, pq, C, V, C, G, feat);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_spmm_gxy(const dn_csr* g, const float* x, int64_t V, int C, float* gxy, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (C != 128 && C != 256) return DN_ERR_UNSUPPORTED;
  const float2* vals = reinterpret_cast<const float2*>(g->vals);
  const unsigned ctas = (unsigned)((V + GB_ROWS - 1) / GB_ROWS);
  // (measured, tools/gf_check.py: streaming stores change nothing, 4 CTAs / SM with 64 registers is 5 % slower)
  if (C == 128) spmm_gxy_blk_kernel<1><<<ctas, 256, 0, st>>>(g->rowptr, g->colidx, vals, x, V, gxy);
  else spmm_gxy_blk_kernel<2><<<ctas, 256, 0, st>>>(g->rowptr, g->colidx, vals, x, V, gxy);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_features_bwd_local(const dn_csr* g, const float* xd, const float* pq, const float* feat,
                              const float* dfeat, int rotations, int64_t V, int C, float* U, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (C % 4) return DN_ERR_UNSUPPORTED;
  const int G = pick_group(C);
  const int64_t warps = (V + (32 / G) - 1) / (32 / G);
  const unsigned blocks = (unsigned)((warps * 32 + 255) / 256);
  const float2* vals = reinterpret_cast<const float2*>(g->vals);
  if (rotations)
    features_bwd_local_kernel<true><<<blocks, 256, 0, st>>>(g->rowptr, g->colidx, vals, xd, pq, 2 * C, feat, dfeat,
                                                             V, C, G, U);
  else
    features_bwd_local_kernel<false><<<blocks, 256, 0, st>>>(g->rowptr, g->colidx, vals, xd, pq, C, feat, dfeat, V,
                                                              C, G, U);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_features_bwd_transpose(const dn_csr* gt, const float* U, int rotations, int64_t V, int C, float* dxd,
                                  float* dP, float* dQ, int64_t ld_pq, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (C % 4) return DN_ERR_UNSUPPORTED;
  const int G = pick_group(C);
  const int64_t warps = (V + (32 / G) - 1) / (32 / G);
  const unsigned blocks = (unsigned)((warps * 32 + 255) / 256);
  const float2* vals = reinterpret_cast<const float2*>(gt->vals);
  if (rotations)
    features_bwd_transpose_kernel<true><<<blocks, 256, 0, st>>>(gt->rowptr, gt->colidx, vals, U, V, C, G, dxd, dP, dQ, ld_pq);
  else
    features_bwd_transpose_kernel<false><<<blocks, 256, 0, st>>>(gt->rowptr, gt->colidx, vals, U, V, C, G, dxd, dP, dQ, ld_pq);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_deinterleave_vc2(const float* vc2, int64_t V, int C, float* g01, cudaStream_t st) {
  const int64_t n = V * C;
  if (n <= 0) return DN_OK;
  deinterleave_vc2_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(reinterpret_cast<const float2*>(vc2), V, C, g01);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int launch_complex_dots_tanh(const float* g01, const float* b01, int64_t V, int C, float* out, cudaStream_t st) {
  const int64_t n = V * C;
  if (n <= 0) return DN_OK;
  complex_dots_tanh_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g01, b01, V, C, out);
  DN_LAUNCH_CHECK();
  return DN_OK;
}
