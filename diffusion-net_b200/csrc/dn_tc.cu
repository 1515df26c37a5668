// tcgen05 tensor-core engine (sm_100a): the dense contractions of the DiffusionNetBlock path.
//
//   tc_rows_chain       fused chain of affine layers over 128-vertex row tiles
//                       (from_basis [+ complex-linear P|Q], MiniMLP + skip)      layers.py:56-67,229-239
//   tc_to_basis_partial split-V  Phi^T (M x)  with the 128x128 accumulator in TMEM   geometry.py:572-583
//
// Arithmetic: kind::tf32 MMAs with fp32 accumulation in TMEM.  "3x" mode splits every operand
// x = hi + lo (both exactly TF32) and issues lo*hi + hi*lo + hi*hi, recovering fp32-grade
// products; "1x" mode issues hi*hi only.
//
// Data movement: weights are pre-split and pre-laid-out in the UMMA canonical (no-swizzle,
// K-major) layout by a small pack kernel and streamed per K-chunk with bulk TMA copies
// (cp.async.bulk + mbarrier complete_tx).  Activations come from HBM (coalesced float4 loads)
// or from the previous layer's TMEM accumulator, are split in registers and stored straight
// into the canonical layout; a producer/consumer mbarrier ring hands K-chunks to the single
// MMA-issuing thread.
#include "dn_internal.h"
#include "dn_tc_ptx.cuh"
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

namespace {

using namespace tc;

constexpr int KC = 16;                          // k-elements per pipeline chunk (2 MMA k-steps of 8)
constexpr int TILE_M = 128;                     // vertex rows per tile == UMMA M
constexpr int NSA = 3;                          // activation-operand ring depth
constexpr int A_IMG = TILE_M * KC * 4;          // 8 KiB: one hi (or lo) A chunk image
constexpr int A_STAGE = 2 * A_IMG;              // hi + lo
constexpr int B_BYTES = 65536;                  // weight ring: 4 stages at N<=128, 2 stages at N=256
constexpr int A_LBO = (TILE_M / 8) * 128;       // 2048 B between k-groups (4 elements) of A
constexpr int CHAIN_THREADS = 320;              // warp0 TMA, warp1 MMA, warps 2..9 workers (2 warpgroups)
constexpr int CHAIN_SMEM = NSA * A_STAGE + B_BYTES + 256;   // 114,944 B: two CTAs fit one SM

struct TcLayer {
  const float* wpack;
  const float* bias;
  const float* residual;
  int64_t ld_res;
  const float* row_scale;
  float* out;
  int64_t ld_out;
  int K, N, relu;
};

struct TcChainParams {
  DnRowsSrc src;
  TcLayer layer[DN_MAX_LAYERS];
  int n_layers;
  int passes;
  int nmax;       // 128 or 256: widest layer (sizes the weight stages and the TMEM buffers)
  int64_t V;
  long long* trace;   // optional (tools/trace_chain.py): per-warp (event, clock64) pairs of CTA 0
  // TMEM plan of the TMEM-A kernel: accumulator column of buffer 0/1, number of buffers, first column and
  // depth (4 or 8) of the activation ring
  int acc_col[2], nbuf, a_col0, nsa;
  int ts_split;   // 1: loader / epilogue warpgroups with a split activation ring; 0: all warpgroups do both
};

// ---------------------------------------------------------------------------------------------
// weight pack:  W -> [chunk][hi | lo][ (k/4)*N*16B + (n/8)*128B + (n%8)*16B + (k%4)*4B ]
// ---------------------------------------------------------------------------------------------
struct PackJob {
  const float* W;
  const float* W2;
  float* dst;
  int64_t ldw;
  int n_split, w_trans, K, N, blk0, fmt;
  // rot_C > 0: the matrix is the complex-linear map of SpatialGradientFeatures (layers.py:121-123) applied to
  // [gX | gY] (K = 2 * rot_C) for channels [rot_ch0, rot_ch0 + N/2):  rows n < N/2 give Bre = A_re gX - A_im gY, rows
  // n >= N/2 give Bim = A_im gX + A_re gY   (W = A_re, W2 = A_im, both (rot_C, rot_C) with row stride ldw)
  int rot_C, rot_ch0;
};
struct PackJobs {
  PackJob j[DN_MAX_LAYERS];
  int n, kc;
  // optional: job 0's matrix is the spectral multiplier S[k][n] = exp(-evals[k] * max(t[n], 1e-8)) * sum_p partial[p][k][n]
  // (layers.py:48-49, 62-64), formed here instead of by a separate launch; the clamped time is written back in place
  const float* sp_partial;
  const float* sp_evals;
  float* sp_time;
  int sp_P, sp_clamp;
};

// one weight element -> its place in the tensor-core layout `fmt` (DnLayer::pack_fmt)
__device__ __forceinline__ void pack_store(float* dst, int fmt, int kc, int N, int k, int n, float w) {
  if (fmt == 2) {
    // bf16, 64-wide stages, K-major canonical (no swizzle): k-group (8 elements) stride N * 16 B, 8-row group stride
    // 128 B, row stride 16 B  (rows_chain16_kernel)
    const int st = k >> 6, kk = k & 63;
    char* base = reinterpret_cast<char*>(dst) + (int64_t)st * N * 128;
    *reinterpret_cast<__nv_bfloat16*>(base + (int64_t)(kk >> 3) * N * 16 + (int64_t)(n >> 3) * 128 + (n & 7) * 16 +
                                      (kk & 7) * 2) = __float2bfloat16_rn(w);
    return;
  }
  float hi, lo;
  split_tf32(w, hi, lo);
  if (fmt == 1) {
    // 32-wide stage = [tf32 hi image: 8 k-groups of 4 | bf16 image: 4 k-groups of 8 of bf16(hi), then 4 of bf16(lo)],
    // both K-major canonical (no swizzle): k-group stride N * 16 B, 8-row group stride 128 B, row stride 16 B
    const int st = k >> 5, kk = k & 31;
    char* base = reinterpret_cast<char*>(dst) + (int64_t)st * N * 256;
    const int64_t rowoff = (int64_t)(n >> 3) * 128 + (n & 7) * 16;
    *reinterpret_cast<float*>(base + (int64_t)(kk >> 2) * N * 16 + rowoff + (kk & 3) * 4) = hi;
    char* b16 = base + (int64_t)N * 128;
    *reinterpret_cast<__nv_bfloat16*>(b16 + (int64_t)(kk >> 3) * N * 16 + rowoff + (kk & 7) * 2) = __float2bfloat16_rn(hi);
    *reinterpret_cast<__nv_bfloat16*>(b16 + (int64_t)(4 + (kk >> 3)) * N * 16 + rowoff + (kk & 7) * 2) =
        __float2bfloat16_rn(w - hi);
    return;
  }
  const int chunk = k / kc, kk = k % kc;
  const int64_t img = (int64_t)N * kc;   // floats per image
  const int64_t off = (int64_t)chunk * 2 * img + (int64_t)(kk >> 2) * (N * 4) + (n >> 3) * 32 + (n & 7) * 4 + (kk & 3);
  dst[off] = hi;
  dst[off + img] = lo;
}

// all weight matrices of a block forward in one launch (blocks are assigned to jobs by blk0)
__global__ void pack_weights_kernel(const __grid_constant__ PackJobs jobs) {
  int ji = 0;
#pragma unroll
  for (int i = 1; i < DN_MAX_LAYERS; ++i)
    if (i < jobs.n && (int)blockIdx.x >= jobs.j[i].blk0) ji = i;
  const PackJob& J = jobs.j[ji];
  const int K = J.K, N = J.N, kc = jobs.kc;
  int n, k;
  float w;
  if (ji == 0 && jobs.sp_partial) {
    // spectral job: a block = 32 consecutive elements (n fastest: coalesced) x 8 slices of the P partial sums, so the
    // ~10 MB of partials are read with many loads in flight (one thread per element was 19 us at K = C = 128)
    __shared__ float red[8][33];
    const int e = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int idx = ((int)blockIdx.x - J.blk0) * 32 + e;
    float acc = 0.f;
    if (idx < K * N) {
      const float* pp = jobs.sp_partial + idx;
      const int64_t stride = (int64_t)K * N;
      for (int q = sl; q < jobs.sp_P; q += 8) acc += pp[(int64_t)q * stride];
    }
    red[sl][e] = acc;
    __syncthreads();
    if (sl != 0 || idx >= K * N) return;
    k = idx / N; n = idx % N;
    const float sum = ((red[0][e] + red[1][e]) + (red[2][e] + red[3][e])) + ((red[4][e] + red[5][e]) + (red[6][e] + red[7][e]));
    const float t = fmaxf(jobs.sp_time[n], 1e-8f);         // torch.clamp(t, min=1e-8)
    w = expf(-(jobs.sp_evals[k] * t)) * sum;
    if (jobs.sp_clamp && k == K - 1) jobs.sp_time[n] = t;   // (idempotent for the other readers of t[n])
  } else {
    const int idx = ((int)blockIdx.x - J.blk0) * blockDim.x + threadIdx.x;
    if (idx >= K * N) return;
    n = idx / K; k = idx % K;
    if (J.rot_C > 0) {
      const int nh = N >> 1, Cc = J.rot_C;
      const bool im = n >= nh;
      const int64_t ch = J.rot_ch0 + (im ? n - nh : n);
      if (k < Cc) w = im ? J.W2[ch * J.ldw + k] : J.W[ch * J.ldw + k];
      else w = im ? J.W[ch * J.ldw + (k - Cc)] : -J.W2[ch * J.ldw + (k - Cc)];
    } else if (J.w_trans) w = (J.W2 && k >= J.n_split) ? J.W2[(int64_t)(k - J.n_split) * J.ldw + n] : J.W[(int64_t)k * J.ldw + n];
    else if (J.W2 && n >= J.n_split) w = J.W2[(int64_t)(n - J.n_split) * J.ldw + k];
    else w = J.W[(int64_t)n * J.ldw + k];
  }
  pack_store(J.dst, J.fmt, kc, N, k, n, w);
}

// mesh batches: the spectral multiplier of every mesh, packed as layer-0 weights of the from_basis chain
//   S_b[k][n] = exp(-evals[b][k] * max(t[n], 1e-8)) * sum_{p in CTAs of mesh b} partial[p][k][n]     (layers.py:48-49, 62-64)
// grid (ceil(K*N/32), n_meshes), 256 threads: 32 consecutive elements x 8 slices of the partial sums per block.
// x_spec_out (optional, [n_meshes][K][N]): the reduced, unscaled coefficients of every mesh (saved for the backward pass)
__global__ void spectral_pack_batched_kernel(const float* __restrict__ partial, const int32_t* __restrict__ mesh_cta_begin,
                                             const float* __restrict__ evals, float* time, int K, int N, int fmt, int kc,
                                             float* dst, int64_t dst_stride_floats, int clamp, float* __restrict__ x_spec_out) {
  __shared__ float red[8][33];
  const int b = blockIdx.y;
  const int e = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int idx = (int)blockIdx.x * 32 + e;
  const int p0 = mesh_cta_begin[b], p1 = mesh_cta_begin[b + 1];
  float acc = 0.f;
  if (idx < K * N) {
    const float* pp = partial + idx;
    const int64_t stride = (int64_t)K * N;
    for (int q = p0 + sl; q < p1; q += 8) acc += pp[(int64_t)q * stride];
  }
  red[sl][e] = acc;
  __syncthreads();
  if (sl != 0 || idx >= K * N) return;
  const int k = idx / N, n = idx % N;
  const float sum = ((red[0][e] + red[1][e]) + (red[2][e] + red[3][e])) + ((red[4][e] + red[5][e]) + (red[6][e] + red[7][e]));
  const float t = fmaxf(time[n], 1e-8f);
  const float w = expf(-(evals[(int64_t)b * K + k] * t)) * sum;
  pack_store(dst + (int64_t)b * dst_stride_floats, fmt, kc, N, k, n, w);
  if (x_spec_out) x_spec_out[(int64_t)b * K * N + idx] = sum;
  // the in-place clamp of the reference: written back by mesh 0 only, after every reader of t[n] in this launch has at
  // worst read either value (max(t, 1e-8) is idempotent)
  if (clamp && b == 0 && k == K - 1) time[n] = t;
}

// mesh batches, backward of the spectral multiplier (the batched form of spectral_bwd_kernel):
//   Gs_b[k][n] = sum_{p in CTAs of mesh b} partial[p][k][n]   (= Phi_b^T g_b),
//   dS_b = exp(-evals[b][k] t[n]) * Gs_b   packed as mesh b's layer-0 weights of the from_basis chain,
//   dt_part[b * gridDim.y + kg][n] = sum over the DN_SPEC_BWD_KROWS rows k of group kg of Gs_b * (-lambda) * E * x_spec_b.
// grid (ceil(N/32), ceil(K/DN_SPEC_BWD_KROWS), n_meshes), 256 threads: 32 consecutive columns x 8 slices of the partials.
// Every sum runs in a fixed order (no atomics): the result does not depend on scheduling.
__global__ void spectral_bwd_pack_batched_kernel(const float* __restrict__ partial, const int32_t* __restrict__ mesh_cta_begin,
                                                 const float* __restrict__ evals, const float* __restrict__ time,
                                                 const float* __restrict__ x_spec, int K, int N, int fmt, int kc, float* dst,
                                                 int64_t dst_stride_floats, float* __restrict__ dt_part) {
  __shared__ float red[8][33];
  const int b = blockIdx.z, kg = blockIdx.y;
  const int e = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int n = (int)blockIdx.x * 32 + e;
  const int p0 = mesh_cta_begin[b], p1 = mesh_cta_begin[b + 1];
  const int64_t stride = (int64_t)K * N;
  const float t = n < N ? fmaxf(time[n], 1e-8f) : 0.f;
  float dt = 0.f;
  for (int i = 0; i < DN_SPEC_BWD_KROWS; ++i) {
    const int k = kg * DN_SPEC_BWD_KROWS + i;
    const bool live = k < K && n < N;
    float acc = 0.f;
    if (live) {
      const float* pp = partial + (int64_t)k * N + n;
      for (int q = p0 + sl; q < p1; q += 8) acc += pp[(int64_t)q * stride];
    }
    red[sl][e] = acc;
    __syncthreads();
    if (sl == 0 && live) {
      const float g = ((red[0][e] + red[1][e]) + (red[2][e] + red[3][e])) + ((red[4][e] + red[5][e]) + (red[6][e] + red[7][e]));
      const float lam = evals[(int64_t)b * K + k];
      const float ex = expf(-(lam * t));
      pack_store(dst + (int64_t)b * dst_stride_floats, fmt, kc, N, k, n, ex * g);
      dt += g * (-lam) * ex * x_spec[(int64_t)b * stride + (int64_t)k * N + n];
    }
    __syncthreads();
  }
  if (sl == 0 && n < N) dt_part[((int64_t)b * gridDim.y + kg) * N + n] = dt;
}

// grad_time[n] += sum_r dt_part[r][n] in a fixed order.  grid ceil(N/32), 1024 threads: 32 columns x 32 row slices
__global__ void grad_time_reduce_kernel(const float* __restrict__ dt_part, int rows, int N, float* __restrict__ grad_time) {
  __shared__ float red[32][33];
  const int e = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int n = (int)blockIdx.x * 32 + e;
  float s = 0.f;
  if (n < N)
    for (int r = sl; r < rows; r += 32) s += dt_part[(int64_t)r * N + n];
  red[sl][e] = s;
  __syncthreads();
  if (sl != 0 || n >= N) return;
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) tot += red[i][e];
  grad_time[n] += tot;
}

// ---------------------------------------------------------------------------------------------
// helpers shared by the worker warps
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void store_split4(uint8_t* a_hi, uint8_t* a_lo, uint32_t byte_off, float4 v, int passes) {
  // hi = rna_tf32(x); lo = x - hi is exact in fp32 and the tensor core reads only its top 19 bits
  float4 h, l;
  split_tf32_fast(v.x, h.x, l.x);
  split_tf32_fast(v.y, h.y, l.y);
  split_tf32_fast(v.z, h.z, l.z);
  split_tf32_fast(v.w, h.w, l.w);
  *reinterpret_cast<float4*>(a_hi + byte_off) = h;
  if (passes == 3) *reinterpret_cast<float4*>(a_lo + byte_off) = l;
}

#define DN_TRACE_MAX 4096
#define DN_TRACE(ev)                                                                  \
  do {                                                                                \
    if (p.trace && blockIdx.x == 0 && lane == 0 && tr_n < DN_TRACE_MAX) {             \
      p.trace[((int64_t)warp * DN_TRACE_MAX + tr_n) * 2] = (ev);                      \
      p.trace[((int64_t)warp * DN_TRACE_MAX + tr_n) * 2 + 1] = clock64();             \
      ++tr_n;                                                                         \
    }                                                                                 \
  } while (0)

// ---------------------------------------------------------------------------------------------
// fused affine chain over 128-row tiles
//
// Two CTAs are co-resident per SM (320 threads, <=113 KB smem, 256 TMEM columns each): while one
// CTA sits in a layer boundary (accumulator drain -> next operand chunks) the other keeps the
// tensor pipe busy.  Per CTA: warp 0 streams weight chunks with bulk TMA (and L2-prefetches the
// next tile's rows), warp 1 issues the MMAs, warps 2..9 (two warpgroups, alternating K-chunks)
// build operand chunks (from HBM/L2 for layer 0, from the TMEM accumulator for chained layers)
// and run the epilogues.  Every role is latency-bound per chunk, so throughput comes from having
// many chunks in flight (2 CTAs x 2 warpgroups) and from keeping the per-chunk instruction
// streams short (incremental ring counters, descriptor templates, one cvt per split).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CHAIN_THREADS, 2) rows_chain_kernel(const __grid_constant__ TcChainParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smA = smem;
  uint8_t* smB = smem + NSA * A_STAGE;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSA * A_STAGE + B_BYTES);
  // bars: full[NSA] empty[NSA] d_full[2] d_empty[2].  One full/empty pair per pipeline stage covers both the
  // activation chunk (4 worker-warp arrivals) and the weight chunk (1 arrive.expect_tx + TMA bytes): the MMA
  // warp waits once and commits once per K-chunk.
  const uint32_t full = smem_u32(bars), empty = smem_u32(bars + NSA);
  const uint32_t d_full = smem_u32(bars + 2 * NSA), d_empty = smem_u32(bars + 2 * NSA + 2);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NSA + 4);

  const int nmax = p.nmax;                                  // 128 or 256: widest layer
  const uint32_t b_stage = 2u * (uint32_t)nmax * KC * 4;    // hi + lo weight chunk (16 or 32 KiB)
  const uint32_t NS = (nmax == 128) ? (uint32_t)NSA : 2u;   // pipeline depth (A and B rings alike)
  const uint32_t nbuf = 256u / (uint32_t)nmax;              // 2 or 1 accumulator buffers in TMEM

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int tr_n = 0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSA; ++i) { mbar_init(full + 8 * i, 5); mbar_init(empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(d_full + 8 * i, 1); mbar_init(d_empty + 8 * i, 8); }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc<256>(smem_u32(tmem_slot));
  // biases of every layer are staged once in the unused tail of the weight ring (N<=128 chains use 48 of
  // its 64 KiB): the epilogues read them with broadcast LDS instead of per-chunk global loads
  float* sbias = reinterpret_cast<float*>(smB + 3 * 16384);
  const bool bias_in_smem = (nmax == 128);
  if (bias_in_smem)
    for (int i = threadIdx.x; i < p.n_layers * 128; i += blockDim.x) {
      const int l = i >> 7, n = i & 127;
      sbias[i] = (p.layer[l].bias && n < p.layer[l].N) ? __ldg(p.layer[l].bias + n) : 0.f;
    }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int L = p.n_layers;
  const int64_t ntiles = (p.V + TILE_M - 1) / TILE_M;

  if (warp == 0) {
    // ===================== weight producer (bulk TMA; warp-uniform, one elected lane issues) =====
    uint32_t s = 0, ph = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      for (int l = 0; l < L; ++l) {
        const int N = p.layer[l].N, nch = p.layer[l].K / KC;
        const uint32_t img_bytes = (uint32_t)N * KC * 4;
        const uint32_t bytes = p.passes == 3 ? 2 * img_bytes : img_bytes;
        const float* wsrc = p.layer[l].wpack;
        for (int c = 0; c < nch; ++c) {
          DN_TRACE(30);
          mbar_wait(empty + 8 * s, ph ^ 1);
          DN_TRACE(31);
          if (elect_one()) {
            mbar_arrive_expect_tx(full + 8 * s, bytes);
            tma_bulk_g2s(smem_u32(smB + s * b_stage), wsrc + (int64_t)c * 2 * N * KC, bytes, full + 8 * s);
          }
          __syncwarp();
          if (++s == NS) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-uniform loop; one elected lane issues) ==============
    // descriptor = template (LBO | SBO | version) + (smem address >> 4); k-steps / lo images are
    // constant increments of the address field
    const uint64_t tmplA = make_desc(0, A_LBO, 128);
    const uint32_t smA_u = smem_u32(smA) >> 4, smB_u = smem_u32(smB) >> 4;
    uint32_t sa = 0, pa = 0, g = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int l = 0; l < L; ++l, ++g) {
        const int N = p.layer[l].N, nch = p.layer[l].K / KC;
        const uint32_t idesc = make_idesc_tf32(TILE_M, N);
        const uint32_t buf = (nbuf == 2) ? (g & 1) : 0, use = (nbuf == 2) ? (g >> 1) : g;
        const uint32_t d_tmem = tmem_base + buf * (uint32_t)nmax;
        const uint32_t b_lbo = (uint32_t)N * 16;
        const uint64_t tmplB = make_desc(0, b_lbo, 128);
        const uint32_t b_img_u = ((uint32_t)N * KC * 4) >> 4, b_ks_u = (2 * b_lbo) >> 4;
        if (use > 0) {   // the epilogue of the previous user of this accumulator buffer must be done
          mbar_wait(d_empty + 8 * buf, (use - 1) & 1);
          tc_fence_after();
        }
        for (int c = 0; c < nch; ++c) {
          DN_TRACE(20);
          mbar_wait(full + 8 * sa, pa);
          DN_TRACE(21);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t dah = tmplA + (smA_u + sa * (A_STAGE >> 4));
            const uint64_t dbh = tmplB + (smB_u + sa * (b_stage >> 4));
#pragma unroll
            for (int ks = 0; ks < KC / 8; ++ks) {
              const uint64_t a_h = dah + ks * ((2 * A_LBO) >> 4), b_h = dbh + ks * b_ks_u;
              const uint32_t acc = (c | ks) ? 1u : 0u;
              if (p.passes == 3) {
                mma_tf32_ss(d_tmem, a_h + (A_IMG >> 4), b_h, idesc, acc);
                mma_tf32_ss(d_tmem, a_h, b_h + b_img_u, idesc, 1u);
                mma_tf32_ss(d_tmem, a_h, b_h, idesc, 1u);
              } else {
                mma_tf32_ss(d_tmem, a_h, b_h, idesc, acc);
              }
            }
            mma_commit(empty + 8 * sa);
            if (c + 1 == nch) mma_commit(d_full + 8 * buf);
          }
          __syncwarp();
          DN_TRACE(22);
          if (++sa == NS) { sa = 0; pa ^= 1; }
        }
      }
  } else {
    // ===================== workers: A-chunk producers + epilogue =====================
    const int wg = (warp - 2) >> 2;           // K-chunk parity this warpgroup owns
    const int quarter = warp & 3;             // TMEM lane quarter this warp may access (rows 32q..32q+31)
    const int rl = lane & 7, kg = lane >> 3;  // conversion mapping: 8 rows x 4 k-groups per warp step
    uint32_t ci = 0, g = 0;
    const int nch0 = p.layer[0].K / KC;
    // byte offset of this lane's 16-byte slot inside an operand image, conversion mapping
    const uint32_t cv_off = kg * A_LBO + (4 * quarter) * 128 + rl * 16;     // + it * 128
    // per-tile row pointers of this lane (one per source); a chunk load is then pointer + column offset
    const float* rowp[DN_MAX_SRC];
    int64_t rem_rows = 0;
    auto set_tile = [&](int64_t row0_) {
      const int64_t rfirst = row0_ + 32 * quarter + rl;
      rem_rows = p.V - rfirst;
#pragma unroll
      for (int q = 0; q < DN_MAX_SRC; ++q)
        rowp[q] = (q < p.src.nsrc) ? p.src.ptr[q] + rfirst * p.src.ld[q] + 4 * kg : nullptr;
    };
    auto load_chunk = [&](int c, float4* r) {
      int k0 = c * KC, s = 0;
      while (s + 1 < p.src.nsrc && k0 >= p.src.width[s]) { k0 -= p.src.width[s]; ++s; }
      const float* base = (s == 0 ? rowp[0] : (s == 1 ? rowp[1] : rowp[2])) + k0;
      const int64_t st8 = 8 * p.src.ld[s];
#pragma unroll
      for (int it = 0; it < 4; ++it)
        r[it] = (8 * it < rem_rows) ? __ldg(reinterpret_cast<const float4*>(base + it * st8))
                                    : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    auto store_chunk = [&](uint32_t cidx, const float4* r) {
      const uint32_t s = cidx % NS, ph = (cidx / NS) & 1;
      DN_TRACE(1);
      mbar_wait(empty + 8 * s, ph ^ 1);
      DN_TRACE(2);
      uint8_t* a_hi = smA + s * A_STAGE + cv_off;
#pragma unroll
      for (int it = 0; it < 4; ++it)
        store_split4(a_hi, a_hi + A_IMG, it * 128, r[it], p.passes);
      DN_TRACE(3);
      fence_proxy_async();
      __syncwarp();
      DN_TRACE(4);
      if (lane == 0) mbar_arrive(full + 8 * s);
      DN_TRACE(5);
    };
    float4 r[4];
    if ((int64_t)blockIdx.x < ntiles) {
      set_tile((int64_t)blockIdx.x * TILE_M);
      if (wg < nch0) load_chunk(wg, r);
    }
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int64_t row0 = tile * TILE_M;
      for (int l = 0; l < L; ++l, ++g) {
        const TcLayer& Lr = p.layer[l];
        const int nch = Lr.K / KC;
        if (l == 0) {
          for (int c = wg; c < nch; c += 2) {
            store_chunk(ci + c, r);
            if (c + 2 < nch) load_chunk(c + 2, r);
          }
          const int64_t nt = tile + gridDim.x;   // first chunk of the next tile: hidden behind the epilogues
          if (nt < ntiles) {
            set_tile(nt * TILE_M);
            if (wg < nch0) load_chunk(wg, r);
          }
        }
        const uint32_t ci_next = ci + nch;
        // ---- epilogue of layer l (and operand production for layer l+1)
        const bool has_next = (l + 1 < L);
        const int64_t row = row0 + 32 * quarter + lane;
        const int rr_ = 32 * quarter + lane;
        const uint32_t ep_off = (rr_ >> 3) * 128 + (rr_ & 7) * 16;
        const int nco = Lr.N / KC;
        const bool has_res = Lr.residual != nullptr;
        const uint32_t buf = (nbuf == 2) ? (g & 1) : 0, use = (nbuf == 2) ? (g >> 1) : g;
        auto load_res = [&](int c, float4* q) {
          const float4* rp = reinterpret_cast<const float4*>(Lr.residual + row * Lr.ld_res + c * KC);
#pragma unroll
          for (int j = 0; j < 4; ++j) q[j] = (row < p.V) ? __ldg(rp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        float4 res[4];
        if (has_res && wg < nco) load_res(wg, res);     // requested before waiting for the accumulator
        const float rs = (Lr.row_scale && row < p.V) ? __ldg(Lr.row_scale + row) : 1.f;
        DN_TRACE(10);
        mbar_wait(d_full + 8 * buf, use & 1);
        DN_TRACE(11);
        tc_fence_after();
        const uint32_t d_lane = tmem_base + ((uint32_t)(32 * quarter) << 16) + buf * (uint32_t)nmax;
        for (int c = wg; c < nco; c += 2) {
          float v[16];
          tmem_ld16(d_lane + c * KC, v);
          DN_TRACE(12);
          const int n0 = c * KC;
          if (Lr.bias) {
            const float4* bp = bias_in_smem ? reinterpret_cast<const float4*>(sbias + l * 128 + n0)
                                            : reinterpret_cast<const float4*>(Lr.bias + n0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = bp[j];
              v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
            }
          }
          if (Lr.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          if (Lr.row_scale) {
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] *= rs;
          }
          if (has_res) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              v[4 * j] += res[j].x; v[4 * j + 1] += res[j].y; v[4 * j + 2] += res[j].z; v[4 * j + 3] += res[j].w;
            }
            if (c + 2 < nco) load_res(c + 2, res);
          }
          DN_TRACE(13);
          if (Lr.out && row < p.V) {
            float4* op = reinterpret_cast<float4*>(Lr.out + row * Lr.ld_out + n0);
#pragma unroll
            for (int j = 0; j < 4; ++j) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          }
          DN_TRACE(14);
          if (has_next) {
            const uint32_t cidx = ci_next + c, s = cidx % NS, ph = (cidx / NS) & 1;
            mbar_wait(empty + 8 * s, ph ^ 1);
            DN_TRACE(15);
            uint8_t* a_hi = smA + s * A_STAGE + ep_off;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              store_split4(a_hi, a_hi + A_IMG, j * A_LBO,
                           make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]), p.passes);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(full + 8 * s);
            DN_TRACE(16);
          }
        }
        // accumulator buffer drained: hand it back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(d_empty + 8 * buf);
        ci = ci_next;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) tmem_dealloc<256>(tmem_base);
}

// ---------------------------------------------------------------------------------------------
// fused affine chain, activations in TMEM (tcgen05.mma with the A operand read from tensor memory)
//
// The smem-operand kernel above moves ~80 KB through shared memory per 16-wide K-chunk (MMA reads of the
// hi/lo activation and weight images, the operand stores, the weight TMA writes) and its trace shows every
// MIO operation (STS, fence.proxy.async, mbarrier, LDG/STG issue) queueing behind that traffic.  Here the
// activation chunks live in TMEM: workers write x = hi + lo with tcgen05.st (one lane per row, the same
// lane<->row mapping tcgen05.ld gives the epilogue, so no transposes and no bank conflicts), the MMA reads A
// from TMEM and only the weight chunks stay in shared memory (40 KB per chunk).  TMEM: columns [0,256)
// accumulators (2 x 128 ping-pong, or 1 x 256), [256,512) an 8-stage ring of (hi16 | lo16) column blocks.
// One CTA per SM: warp 0 weight TMA, warp 1 MMA, warps 2..17 = four worker warpgroups (K-chunk c -> c % 4).
// ---------------------------------------------------------------------------------------------
constexpr int TS_THREADS = 576;
constexpr int TS_NSA = 8;                    // activation stages in TMEM
constexpr int TS_BIAS_FLOATS = DN_MAX_LAYERS * 256;
constexpr int TS_BBYTES = 131072;            // weight ring: 8 stages at N<=128, 4 at N=256
constexpr int TS_SMEM = TS_BBYTES + TS_BIAS_FLOATS * 4 + 512;

__global__ void __launch_bounds__(TS_THREADS, 1) rows_chain_ts_kernel(const __grid_constant__ TcChainParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* smB = smem;
  float* sbias = reinterpret_cast<float*>(smem + TS_BBYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TS_BBYTES + TS_BIAS_FLOATS * 4);
  // bars: a_full[8] a_empty[8] b_full[8] b_empty[8] d_full[2] d_empty[2]
  const uint32_t a_full = smem_u32(bars), a_empty = smem_u32(bars + TS_NSA);
  const uint32_t b_full = smem_u32(bars + 2 * TS_NSA), b_empty = smem_u32(bars + 2 * TS_NSA + 8);
  const uint32_t d_full = smem_u32(bars + 2 * TS_NSA + 16), d_empty = smem_u32(bars + 2 * TS_NSA + 18);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TS_NSA + 20);

  const int nmax = p.nmax;
  const uint32_t b_stage = 2u * (uint32_t)nmax * KC * 4;    // hi + lo weight chunk (16 or 32 KiB)
  const uint32_t nsb = TS_BBYTES / b_stage;                 // 8 or 4
  const uint32_t nbuf = (uint32_t)p.nbuf;                   // 2 or 1 accumulator buffers
  // the activation ring is split in two halves with their own barriers: half 0 holds layer-0 chunks (written by
  // the loader warps, which may run ahead into the next tile), half 1 the chained-layer chunks (written by the
  // epilogue warps).  Each half has a single in-order producer stream, which the mbarrier parity protocol needs.
  // (p.ts_split == 0: one ring, all warpgroups produce in program order.)
  const bool split = p.ts_split != 0;
  const uint32_t nsh = split ? (uint32_t)p.nsa / 2 : (uint32_t)p.nsa;           // stages per ring (half)
  const uint32_t nsh_sh = (nsh == 8) ? 3u : ((nsh == 4) ? 2u : 1u);
  const uint32_t a_col0 = (uint32_t)p.a_col0;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < TS_NSA; ++i) { mbar_init(a_full + 8 * i, 4); mbar_init(a_empty + 8 * i, 1); }
    for (int i = 0; i < 8; ++i) { mbar_init(b_full + 8 * i, 1); mbar_init(b_empty + 8 * i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(d_full + 8 * i, 1); mbar_init(d_empty + 8 * i, p.ts_split ? 8 : 16); }
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc<512>(smem_u32(tmem_slot));
  for (int i = threadIdx.x; i < p.n_layers * 256; i += blockDim.x) {
    const int l = i >> 8, n = i & 255;
    sbias[i] = (p.layer[l].bias && n < p.layer[l].N) ? __ldg(p.layer[l].bias + n) : 0.f;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int L = p.n_layers;
  const int64_t ntiles = (p.V + TILE_M - 1) / TILE_M;

  if (warp == 0) {
    // ===================== weight producer (bulk TMA) =====================
    uint32_t s = 0, ph = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int l = 0; l < L; ++l) {
        const int N = p.layer[l].N, nch = p.layer[l].K / KC;
        const uint32_t img_bytes = (uint32_t)N * KC * 4;
        const uint32_t bytes = p.passes == 3 ? 2 * img_bytes : img_bytes;
        const float* wsrc = p.layer[l].wpack;
        for (int c = 0; c < nch; ++c) {
          mbar_wait(b_empty + 8 * s, ph ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(b_full + 8 * s, bytes);
            tma_bulk_g2s(smem_u32(smB + s * b_stage), wsrc + (int64_t)c * 2 * N * KC, bytes, b_full + 8 * s);
          }
          __syncwarp();
          if (++s == nsb) { s = 0; ph ^= 1; }
        }
      }
  } else if (warp == 1) {
    // ===================== MMA issuer: A from TMEM, B from shared memory =====================
    const uint32_t smB_u = smem_u32(smB) >> 4;
    uint32_t s0 = 0, p0 = 0, s1 = 0, p1 = 0, sb = 0, pb = 0, g = 0;   // ring half 0: layer-0 chunks, half 1: chained
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int l = 0; l < L; ++l, ++g) {
        const int N = p.layer[l].N, nch = p.layer[l].K / KC;
        const uint32_t idesc = make_idesc_tf32(TILE_M, N);
        const uint32_t buf = (nbuf == 2) ? (g & 1) : 0, use = (nbuf == 2) ? (g >> 1) : g;
        const uint32_t d_tmem = tmem_base + (uint32_t)p.acc_col[buf];
        const uint32_t b_lbo = (uint32_t)N * 16;
        const uint64_t tmplB = make_desc(0, b_lbo, 128);
        const uint32_t b_img_u = ((uint32_t)N * KC * 4) >> 4, b_ks_u = (2 * b_lbo) >> 4;
        if (use > 0) {
          mbar_wait(d_empty + 8 * buf, (use - 1) & 1);
          tc_fence_after();
        }
        for (int c = 0; c < nch; ++c) {
          const uint32_t hf = (l == 0 || !split) ? 0u : 1u;
          const uint32_t sa = hf ? nsh + s1 : s0;
          mbar_wait(a_full + 8 * sa, hf ? p1 : p0);
          mbar_wait(b_full + 8 * sb, pb);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t a_hi0 = tmem_base + a_col0 + sa * 32;
            const uint64_t dbh = tmplB + (smB_u + sb * (b_stage >> 4));
#pragma unroll
            for (int ks = 0; ks < KC / 8; ++ks) {
              const uint32_t a_hi = a_hi0 + ks * 8, a_lo = a_hi + 16;
              const uint64_t b_h = dbh + ks * b_ks_u;
              const uint32_t acc = (c | ks) ? 1u : 0u;
              if (p.passes == 3) {
                mma_tf32_ts(d_tmem, a_lo, b_h, idesc, acc);
                mma_tf32_ts(d_tmem, a_hi, b_h + b_img_u, idesc, 1u);
                mma_tf32_ts(d_tmem, a_hi, b_h, idesc, 1u);
              } else {
                mma_tf32_ts(d_tmem, a_hi, b_h, idesc, acc);
              }
            }
            mma_commit(a_empty + 8 * sa);
            mma_commit(b_empty + 8 * sb);
            if (c + 1 == nch) mma_commit(d_full + 8 * buf);
          }
          __syncwarp();
          if (hf) { if (++s1 == nsh) { s1 = 0; p1 ^= 1; } }
          else    { if (++s0 == nsh) { s0 = 0; p0 ^= 1; } }
          if (++sb == nsb) { sb = 0; pb ^= 1; }
        }
      }
  } else {
    // ===================== workers: two LOADER warpgroups + two EPILOGUE warpgroups =====================
    // Loaders only build layer-0 chunks from HBM and are throttled solely by the activation ring, so while the
    // MMA works on a tile's last layer (and the epilogue warps drain it) they already stream the next tile in.
    // Epilogue warps own every accumulator read: bias/ReLU/residual, the output store and the next layer's chunks.
    const int ww = warp - 2;
    const bool is_loader = ww < 8;
    const int par = (ww >> 2) & 1;            // K-chunk parity this warpgroup owns inside its role
    const int quarter = warp & 3;             // TMEM lane quarter: this lane owns tile row 32*quarter + lane
    const int trow = 32 * quarter + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(32 * quarter) << 16);
    // x = hi + lo -> TMEM stage (hi in columns [0,16), lo in [16,32) of the stage), then hand it to the MMA
    auto put_chunk = [&](uint32_t hf, uint32_t idx, const float* x16) {     // idx: running chunk count of that half
      const uint32_t s = hf * nsh + (idx & (nsh - 1)), ph = (idx >> nsh_sh) & 1;
      mbar_wait(a_empty + 8 * s, ph ^ 1);
      tc_fence_after();
      float hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) split_tf32_fast(x16[j], hi[j], lo[j]);
      const uint32_t ta = lane_base + a_col0 + s * 32;
      tmem_st16(ta, hi);
      if (p.passes == 3) tmem_st16(ta + 16, lo);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(a_full + 8 * s);
    };
    if (!split) {
      // ---- unspecialised: all four warpgroups build layer-0 chunks (c % 4) and run the epilogues in program order
      const int wgi = ww >> 2;
      const int nch0 = p.layer[0].K / KC;
      const float* rowp[DN_MAX_SRC];
      bool row_ok = false;
      auto set_tile = [&](int64_t row0_) {
        const int64_t rr = row0_ + trow;
        row_ok = rr < p.V;
#pragma unroll
        for (int q = 0; q < DN_MAX_SRC; ++q) rowp[q] = (q < p.src.nsrc) ? p.src.ptr[q] + rr * p.src.ld[q] : nullptr;
      };
      auto load_chunk = [&](int c, float4* r) {
        int k0 = c * KC, s = 0;
        while (s + 1 < p.src.nsrc && k0 >= p.src.width[s]) { k0 -= p.src.width[s]; ++s; }
        const float4* base = reinterpret_cast<const float4*>((s == 0 ? rowp[0] : (s == 1 ? rowp[1] : rowp[2])) + k0);
#pragma unroll
        for (int j = 0; j < 4; ++j) r[j] = row_ok ? __ldg(base + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      uint32_t ci = 0, g = 0;
      float4 r[4];
      if ((int64_t)blockIdx.x < ntiles) {
        set_tile((int64_t)blockIdx.x * TILE_M);
        if (wgi < nch0) load_chunk(wgi, r);
      }
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * TILE_M;
        for (int l = 0; l < L; ++l, ++g) {
          const TcLayer& Lr = p.layer[l];
          const int nch = Lr.K / KC;
          if (l == 0) {
            for (int c = wgi; c < nch; c += 4) {
              float x16[16];
  #pragma unroll
              for (int j = 0; j < 4; ++j) { x16[4 * j] = r[j].x; x16[4 * j + 1] = r[j].y; x16[4 * j + 2] = r[j].z; x16[4 * j + 3] = r[j].w; }
              if (c + 4 < nch) load_chunk(c + 4, r);       // next chunk's loads fly while this one is converted
              put_chunk(0u, ci + c, x16);
            }
            const int64_t nt = tile + gridDim.x;
            if (nt < ntiles) {
              set_tile(nt * TILE_M);
              if (wgi < nch0) load_chunk(wgi, r);
            }
          }
          const uint32_t ci_next = ci + nch;
          // ---- epilogue of layer l (and operand production for layer l+1)
          const bool has_next = (l + 1 < L);
          const int64_t row = row0 + trow;
          const int nco = Lr.N / KC;
          const bool has_res = Lr.residual != nullptr;
          const uint32_t buf = (nbuf == 2) ? (g & 1) : 0, use = (nbuf == 2) ? (g >> 1) : g;
          auto load_res = [&](int c, float4* q) {
            const float4* rp = reinterpret_cast<const float4*>(Lr.residual + row * Lr.ld_res + c * KC);
  #pragma unroll
            for (int j = 0; j < 4; ++j) q[j] = (row < p.V) ? __ldg(rp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
          };
          float4 res[4];
          if (has_res && wgi < nco) load_res(wgi, res);
          const float rs = (Lr.row_scale && row < p.V) ? __ldg(Lr.row_scale + row) : 1.f;
          mbar_wait(d_full + 8 * buf, use & 1);
          tc_fence_after();
          const uint32_t d_lane = lane_base + (uint32_t)p.acc_col[buf];
          for (int c = wgi; c < nco; c += 4) {
            float v[16];
            tmem_ld16(d_lane + c * KC, v);
            const int n0 = c * KC;
            if (Lr.bias) {
              const float4* bp = reinterpret_cast<const float4*>(sbias + l * 256 + n0);
  #pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 b = bp[j];
                v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
              }
            }
            if (Lr.relu) {
  #pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (Lr.row_scale) {
  #pragma unroll
              for (int j = 0; j < 16; ++j) v[j] *= rs;
            }
            if (has_res) {
  #pragma unroll
              for (int j = 0; j < 4; ++j) {
                v[4 * j] += res[j].x; v[4 * j + 1] += res[j].y; v[4 * j + 2] += res[j].z; v[4 * j + 3] += res[j].w;
              }
              if (c + 4 < nco) load_res(c + 4, res);
            }
            if (Lr.out && row < p.V) {
              float4* op = reinterpret_cast<float4*>(Lr.out + row * Lr.ld_out + n0);
  #pragma unroll
              for (int j = 0; j < 4; ++j) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (has_next) put_chunk(0u, ci_next + c, v);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(d_empty + 8 * buf);
          ci = ci_next;
        }
      }
    } else if (is_loader) {
      const int nch0 = p.layer[0].K / KC;
      const float* rowp[DN_MAX_SRC];
      bool row_ok = false;
      auto set_tile = [&](int64_t row0_) {
        const int64_t rr = row0_ + trow;
        row_ok = rr < p.V;
#pragma unroll
        for (int q = 0; q < DN_MAX_SRC; ++q) rowp[q] = (q < p.src.nsrc) ? p.src.ptr[q] + rr * p.src.ld[q] : nullptr;
      };
      auto load_chunk = [&](int c, float4* r) {     // 16 consecutive floats of this lane's own row
        int k0 = c * KC, s = 0;
        while (s + 1 < p.src.nsrc && k0 >= p.src.width[s]) { k0 -= p.src.width[s]; ++s; }
        const float4* base = reinterpret_cast<const float4*>((s == 0 ? rowp[0] : (s == 1 ? rowp[1] : rowp[2])) + k0);
#pragma unroll
        for (int j = 0; j < 4; ++j) r[j] = row_ok ? __ldg(base + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      auto unpack = [&](const float4* r, float* x16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) { x16[4 * j] = r[j].x; x16[4 * j + 1] = r[j].y; x16[4 * j + 2] = r[j].z; x16[4 * j + 3] = r[j].w; }
      };
      float4 r0[4], r1[4];                      // two chunks of this warpgroup in flight
      uint32_t tbase = 0;                       // running count of layer-0 chunks before this tile
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, tbase += (uint32_t)nch0) {
        set_tile(tile * TILE_M);
        if (par < nch0) load_chunk(par, r0);
        if (par + 2 < nch0) load_chunk(par + 2, r1);
        int c = par;
        while (c < nch0) {
          float x16[16];
          unpack(r0, x16);
          if (c + 4 < nch0) load_chunk(c + 4, r0);
          put_chunk(0u, tbase + c, x16);
          c += 2;
          if (c >= nch0) break;
          unpack(r1, x16);
          if (c + 4 < nch0) load_chunk(c + 4, r1);
          put_chunk(0u, tbase + c, x16);
          c += 2;
        }
      }
    } else {
      uint32_t ci = 0, g = 0;                   // ci: running count of chained-layer chunks
      for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * TILE_M;
        for (int l = 0; l < L; ++l, ++g) {
          const TcLayer& Lr = p.layer[l];
          const bool has_next = (l + 1 < L);
          const int64_t row = row0 + trow;
          const int nco = Lr.N / KC;
          const bool has_res = Lr.residual != nullptr;
          const uint32_t buf = (nbuf == 2) ? (g & 1) : 0, use = (nbuf == 2) ? (g >> 1) : g;
          auto load_res = [&](int c, float4* q) {
            const float4* rp = reinterpret_cast<const float4*>(Lr.residual + row * Lr.ld_res + c * KC);
#pragma unroll
            for (int j = 0; j < 4; ++j) q[j] = (row < p.V) ? __ldg(rp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
          };
          float4 res[4];
          if (has_res && par < nco) load_res(par, res);
          const float rs = (Lr.row_scale && row < p.V) ? __ldg(Lr.row_scale + row) : 1.f;
          mbar_wait(d_full + 8 * buf, use & 1);
          tc_fence_after();
          const uint32_t d_lane = lane_base + (uint32_t)p.acc_col[buf];
          for (int c = par; c < nco; c += 2) {
            float v[16];
            tmem_ld16(d_lane + c * KC, v);
            const int n0 = c * KC;
            if (Lr.bias) {
              const float4* bp = reinterpret_cast<const float4*>(sbias + l * 256 + n0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 b = bp[j];
                v[4 * j] += b.x; v[4 * j + 1] += b.y; v[4 * j + 2] += b.z; v[4 * j + 3] += b.w;
              }
            }
            if (Lr.relu) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
            }
            if (Lr.row_scale) {
#pragma unroll
              for (int j = 0; j < 16; ++j) v[j] *= rs;
            }
            if (has_res) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                v[4 * j] += res[j].x; v[4 * j + 1] += res[j].y; v[4 * j + 2] += res[j].z; v[4 * j + 3] += res[j].w;
              }
              if (c + 2 < nco) load_res(c + 2, res);
            }
            if (Lr.out && row < p.V) {
              float4* op = reinterpret_cast<float4*>(Lr.out + row * Lr.ld_out + n0);
#pragma unroll
              for (int j = 0; j < 4; ++j) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
            if (has_next) put_chunk(1u, ci + c, v);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(d_empty + 8 * buf);
          if (has_next) ci += (uint32_t)nco;          // layer l+1 consumed N_l / KC chained chunks
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) tmem_dealloc<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------
// to_basis, split over V:  partial[cta][k][c] = sum_{v in cta's range} Phi[v][k] * m[v] * x[v][c]
//   A = Phi^T (M = K_eig rows, padded to 128), B = (m x)^T (N = C rows); reduction dim = v.
//   Both operands are transposed on the fly: each lane loads a 4(v) x 4(k) block with float4
//   row loads and writes four 16-byte k-major vectors.  SBO is padded to 144 B so those
//   stores are bank-conflict free.
// ---------------------------------------------------------------------------------------------
constexpr int TB_SBO = 144;
constexpr int TB_LBO = 16 * TB_SBO;          // 16 eight-row groups (128 rows) per k-group
constexpr int TB_IMG = 4 * TB_LBO;           // 4 k-groups (16 v) : 9216 B
constexpr int TB_STAGE = 4 * TB_IMG;         // A hi, A lo, B hi, B lo
constexpr int TB_NOP = 4;                    // operand (UMMA-layout) ring depth
constexpr int TB_NST = 4;                    // raw TMA staging ring depth
constexpr int TB_RAW_HALF = KC * 128 * 4;    // 16 rows x up to 128 floats
constexpr int TB_RAW = 2 * TB_RAW_HALF;      // raw Phi rows + raw x rows
constexpr int TB_THREADS = 576;              // warp0 TMA, warp1 MMA, warps 2..17 converters (two sets of 8)
constexpr int TB_SMEM = TB_NST * TB_RAW + TB_NOP * TB_STAGE + 1024;

struct TcToBasisParams {
  const float* values;   // (V, C)
  const float* basis;    // (V, K)
  const float* mass;     // (V) or null
  float* partial;        // (grid, K, C)
  int64_t V;
  int K, C, passes;
  int64_t chunks_per_cta;
  int64_t ld_values;     // row stride of `values` (floats): == C for a contiguous matrix, > C for a column slice
  int64_t ldp;           // row stride of a partial (floats): partial[cta][k][ldp]
  const int32_t* cta_rows;   // optional device [2 * grid]: the row range [begin, end) CTA i reduces (mesh batches: a CTA
};                           //   never crosses a mesh boundary); null = uniform chunks_per_cta * 16 rows per CTA

// TMEM columns: [0,128) correction terms (lo*hi + hi*lo); [128,256) [256,384) [384,512) three
// round-robin accumulators for hi*hi.  Short, separate accumulation chains keep the truncation
// of the tensor-core accumulator below fp32 noise even for V = 200k.
__global__ void __launch_bounds__(TB_THREADS, 1) to_basis_kernel(const __grid_constant__ TcToBasisParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* raw = smem;
  uint8_t* opr = smem + TB_NST * TB_RAW;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TB_NST * TB_RAW + TB_NOP * TB_STAGE);
  const uint32_t st_full = smem_u32(bars), st_empty = smem_u32(bars + TB_NST);
  const uint32_t op_full = smem_u32(bars + 2 * TB_NST), op_empty = smem_u32(bars + 2 * TB_NST + TB_NOP);
  const uint32_t d_full = smem_u32(bars + 2 * TB_NST + 2 * TB_NOP);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TB_NST + 2 * TB_NOP + 2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < TB_NST; ++i) { mbar_init(st_full + 8 * i, 1); mbar_init(st_empty + 8 * i, 8); }
    for (int i = 0; i < TB_NOP; ++i) { mbar_init(op_full + 8 * i, 8); mbar_init(op_empty + 8 * i, 1); }
    mbar_init(d_full, 1);
    fence_barrier_init();
  }
  // operand rows that no lane writes (k >= K or c >= C inside the 128-row images) must be zero
  for (int i = threadIdx.x; i < TB_NOP * TB_STAGE / 16; i += blockDim.x)
    reinterpret_cast<float4*>(opr)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  fence_proxy_async();
  if (warp == 0) tmem_alloc<512>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // this CTA reduces rows [rb, re) in chunks of KC (the last one may be short)
  int64_t rb, re;
  if (p.cta_rows) {
    rb = p.cta_rows[2 * blockIdx.x];
    re = p.cta_rows[2 * blockIdx.x + 1];
  } else {
    rb = (int64_t)blockIdx.x * p.chunks_per_cta * KC;
    re = rb + p.chunks_per_cta * KC;
    if (re > p.V) re = p.V;
  }
  const int64_t nch = re > rb ? (re - rb + KC - 1) / KC : 0;

  if (warp == 0) {
    // ===== TMA producer: 16 consecutive rows of Phi and of x are contiguous in HBM =====
    for (int64_t c = 0; c < nch; ++c) {
      const uint32_t s = c % TB_NST, ph = (c / TB_NST) & 1;
      mbar_wait(st_empty + 8 * s, ph ^ 1);
      const int64_t v0 = rb + c * KC;
      const int nv = (int)((re - v0) < KC ? (re - v0) : KC);
      const uint32_t ba = (uint32_t)nv * p.K * 4, bb = (uint32_t)nv * p.C * 4;
      if (elect_one()) {
        mbar_arrive_expect_tx(st_full + 8 * s, ba + bb);
        tma_bulk_g2s(smem_u32(raw + s * TB_RAW), p.basis + v0 * p.K, ba, st_full + 8 * s);
        if (p.ld_values == p.C) {
          tma_bulk_g2s(smem_u32(raw + s * TB_RAW + TB_RAW_HALF), p.values + v0 * p.C, bb, st_full + 8 * s);
        } else {   // a column slice of a wider matrix: one copy per row
          for (int j = 0; j < nv; ++j)
            tma_bulk_g2s(smem_u32(raw + s * TB_RAW + TB_RAW_HALF) + (uint32_t)j * p.C * 4, p.values + (v0 + j) * p.ld_values,
                         (uint32_t)p.C * 4, st_full + 8 * s);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===== MMA issuer (warp-uniform loop; one elected lane issues) =====
    const uint32_t idesc = make_idesc_tf32(128, p.C);
    const uint32_t lbo = TB_LBO, sbo = TB_SBO;
    for (int64_t c = 0; c < nch; ++c) {
      const uint32_t s = c % TB_NOP, ph = (c / TB_NOP) & 1;
      mbar_wait(op_full + 8 * s, ph);
      tc_fence_after();
      const uint32_t a_hi = smem_u32(opr + s * TB_STAGE), a_lo = a_hi + TB_IMG, b_hi = a_hi + 2 * TB_IMG,
                     b_lo = a_hi + 3 * TB_IMG;
      const uint32_t d_main = tmem_base + 128 * (1 + (uint32_t)(c % 3));
      if (elect_one()) {
#pragma unroll
        for (int ks = 0; ks < KC / 8; ++ks) {
          const uint32_t o = ks * 2 * TB_LBO;
          const uint64_t dah = make_desc(a_hi + o, lbo, sbo), dbh = make_desc(b_hi + o, lbo, sbo);
          if (p.passes == 3) {
            const uint64_t dal = make_desc(a_lo + o, lbo, sbo), dbl = make_desc(b_lo + o, lbo, sbo);
            mma_tf32_ss(tmem_base, dal, dbh, idesc, (c | ks) ? 1u : 0u);
            mma_tf32_ss(tmem_base, dah, dbl, idesc, 1u);
          }
          mma_tf32_ss(d_main, dah, dbh, idesc, (c >= 3 || ks) ? 1u : 0u);
        }
        mma_commit(op_empty + 8 * s);
        if (c + 1 == nch) mma_commit(d_full);
      }
      __syncwarp();
    }
  } else {
    // ===== converters: two sets of 8 warps alternate chunks (the per-chunk wait->LDS->split->STS->fence->arrive
    // chain is latency-bound, so two chunks are converted concurrently); inside a set warps 0..3 build
    // A = Phi^T and warps 4..7 build B = (m x)^T, 4 vertices each =====
    const int cset = (warp - 2) >> 3;
    const int w = (warp - 2) & 7;
    const bool isB = w >= 4;
    const int vg = w & 3;
    const int width = isB ? p.C : p.K;
    const bool active = 4 * lane < width;
    const bool use_mass = isB && p.mass;
    // mass values are fetched one chunk ahead so their L2/HBM latency is off the per-chunk path
    float mnext[4] = {1.f, 1.f, 1.f, 1.f};
    if (use_mass && nch > 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int64_t v = rb + cset * KC + 4 * vg + j;
        mnext[j] = (v < re) ? __ldg(p.mass + v) : 0.f;
      }
    }
    for (int64_t c = cset; c < nch; c += 2) {
      const int64_t v0 = rb + c * KC + 4 * vg;
      float m[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) m[j] = mnext[j];
      if (use_mass && c + 2 < nch) {
#pragma unroll
        for (int j = 0; j < 4; ++j) mnext[j] = (v0 + 2 * KC + j < re) ? __ldg(p.mass + v0 + 2 * KC + j) : 0.f;
      }
      const uint32_t s = c % TB_NST, ph = (c / TB_NST) & 1;
      mbar_wait(st_full + 8 * s, ph);
      float4 q[4];
      const uint8_t* rp = raw + s * TB_RAW + (isB ? TB_RAW_HALF : 0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        q[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (active && v0 + j < re)
          q[j] = *reinterpret_cast<const float4*>(rp + (size_t)(4 * vg + j) * width * 4 + 16 * lane);
        q[j].x *= m[j]; q[j].y *= m[j]; q[j].z *= m[j]; q[j].w *= m[j];   // (values * massvec), geometry.py:583
      }
      const uint32_t o = c % TB_NOP, po = (c / TB_NOP) & 1;
      mbar_wait(op_empty + 8 * o, po ^ 1);
      if (active) {
        uint8_t* hi = opr + o * TB_STAGE + (isB ? 2 * TB_IMG : 0);
        uint8_t* lo = hi + TB_IMG;
        // transpose the 4(v) x 4(col) block: one 16-byte k-major vector per operand row
        const float col[4][4] = {{q[0].x, q[1].x, q[2].x, q[3].x},
                                 {q[0].y, q[1].y, q[2].y, q[3].y},
                                 {q[0].z, q[1].z, q[2].z, q[3].z},
                                 {q[0].w, q[1].w, q[2].w, q[3].w}};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int mrow = 4 * lane + i;   // operand row (eigen-index k, or channel c)
          store_split4(hi, lo, vg * TB_LBO + (mrow >> 3) * TB_SBO + (mrow & 7) * 16,
                       make_float4(col[i][0], col[i][1], col[i][2], col[i][3]), p.passes);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(op_full + 8 * o);
        mbar_arrive(st_empty + 8 * s);
      }
    }
    // ---- epilogue: sum the TMEM accumulators -> partial[cta][k][c]  (warps 2..5 = 4 lane quarters)
    if (cset == 0 && w < 4) {
      float* out = p.partial + (int64_t)blockIdx.x * p.K * p.ldp;
      const int quarter = warp & 3;
      const int k = 32 * quarter + lane;
      if (nch > 0) {
        mbar_wait(d_full, 0);
        tc_fence_after();
      }
      const uint32_t lane_base = tmem_base + ((uint32_t)(32 * quarter) << 16);
      for (int c0 = 0; c0 < p.C; c0 += 16) {
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.f;
        if (nch > 0) {
          float t[16];
          if (p.passes == 3) tmem_ld16(lane_base + c0, v);
          const int nmain = nch < 3 ? (int)nch : 3;
          for (int b = 0; b < nmain; ++b) {
            tmem_ld16(lane_base + 128 * (1 + b) + c0, t);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] += t[j];
          }
        }
        if (k < p.K) {
          float4* op = reinterpret_cast<float4*>(out + (int64_t)k * p.ldp + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j) op[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 0) tmem_dealloc<512>(tmem_base);
}

long long* g_trace_ptr = nullptr;

// Per-device state: capability, SM count, and whether the >48 KB dynamic shared memory attributes were set on that
// device (function attributes are per device: a process that drives several GPUs needs them on each one).
constexpr int kMaxDev = 64;
struct DevState { int tried, ok, sms; };
DevState g_dev[kMaxDev];

}  // namespace

static int g_trace_skip = 0;   // chain launches to let pass before the traced one
extern "C" void dn_debug_set_trace(void* device_buffer) { g_trace_ptr = static_cast<long long*>(device_buffer); g_trace_skip = 0; }
// trace the k-th (0-based) chain-kernel launch after this call instead of every launch
extern "C" void dn_debug_set_trace_launch(int k) { g_trace_skip = k; }
static long long* take_trace_ptr() {
  if (!g_trace_ptr) return nullptr;
  if (g_trace_skip > 0) { --g_trace_skip; return nullptr; }
  if (g_trace_skip == 0) { g_trace_skip = -1; return g_trace_ptr; }
  return nullptr;   // already used once
}

// declared in dn_chain.cu
int tc_chain3_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers);
int tc_rows_chain3(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int64_t V, int passes, int sm_count,
                   long long* trace, cudaStream_t st);
// declared in dn_chain16.cu (bf16 engine)
int tc_chain16_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers);
int tc_rows_chain16(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int64_t V, int sm_count, cudaStream_t st);

static DevState* cur_dev_state() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDev) {
    cudaGetLastError();
    return nullptr;
  }
  DevState& d = g_dev[dev];
  if (!d.tried) {
    d.tried = 1;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
      cudaGetLastError();
      d.ok = 0;
    } else {
      d.ok = (prop.major == 10) ? 1 : 0;
      d.sms = prop.multiProcessorCount;
      if (d.ok) {
        if (cudaFuncSetAttribute(rows_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CHAIN_SMEM) !=
                cudaSuccess ||
            cudaFuncSetAttribute(rows_chain_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                 cudaSharedmemCarveoutMaxShared) != cudaSuccess ||
            cudaFuncSetAttribute(rows_chain_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TS_SMEM) !=
                cudaSuccess ||
            cudaFuncSetAttribute(to_basis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM) !=
                cudaSuccess) {
          cudaGetLastError();
          d.ok = 0;
        }
      }
    }
    const char* off = getenv("DN_TC_DISABLE");
    if (off && atoi(off)) d.ok = 0;
  }
  return &d;
}

bool tc_supported_device() {
  DevState* d = cur_dev_state();
  return d && d->ok == 1;
}

static bool ts_allowed_env() {
  const char* e = getenv("DN_TC_TS");
  return !e || atoi(e) != 0;
}

// shapes the round-1 kernels (rows_chain_kernel / rows_chain_ts_kernel) take
static int tc_rows_chain_legacy_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers) {
  if (n_layers < 1 || n_layers > DN_MAX_LAYERS) return DN_ERR_UNSUPPORTED;
  int k0 = 0;
  for (int s = 0; s < src.nsrc; ++s) {
    if (src.width[s] % 16 || src.ld[s] % 4 || (reinterpret_cast<uintptr_t>(src.ptr[s]) & 15)) return DN_ERR_UNSUPPORTED;
    k0 += src.width[s];
  }
  if (k0 != layers[0].K) return DN_ERR_UNSUPPORTED;
  for (int l = 0; l < n_layers; ++l) {
    const DnLayer& L = layers[l];
    if (L.K % 16 || L.K < 16 || L.N % 16 || L.N < 16 || L.N > 256) return DN_ERR_UNSUPPORTED;
    if (L.emul || L.relu_mask_src || L.dots_src || L.head_w) return DN_ERR_UNSUPPORTED;
    if (L.bias && (reinterpret_cast<uintptr_t>(L.bias) & 15)) return DN_ERR_UNSUPPORTED;
    if (L.residual && (L.res_scale != 1.f || L.ld_res % 4 || (reinterpret_cast<uintptr_t>(L.residual) & 15)))
      return DN_ERR_UNSUPPORTED;
    if (L.out && (L.ld_out % 4 || (reinterpret_cast<uintptr_t>(L.out) & 15))) return DN_ERR_UNSUPPORTED;
    if (l > 0 && L.K != layers[l - 1].N) return DN_ERR_UNSUPPORTED;
    // a 256-wide accumulator cannot ping-pong with another one; the TMEM-A kernel still fits the two-layer
    // pattern (N0 <= 128 then N1 <= 256: from_basis -> [P|Q]) next to a 4-stage activation ring
    if (L.N > 128 && n_layers > 1 && !(ts_allowed_env() && n_layers == 2 && l == 1 && layers[0].N <= 128))
      return DN_ERR_UNSUPPORTED;
  }
  if (!layers[n_layers - 1].out) return DN_ERR_UNSUPPORTED;
  return DN_OK;
}

int tc_rows_chain_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int passes) {
  if (passes == DN_PASSES_BF16 && tc_chain16_supported(src, layers, n_layers) == DN_OK) return DN_OK;
  if (tc_chain3_supported(src, layers, n_layers) == DN_OK) return DN_OK;
  return tc_rows_chain_legacy_supported(src, layers, n_layers);
}

static bool hybrid_enabled() {
  static int on = -1;
  if (on < 0) {
    const char* e = getenv("DN_TC_HYBRID");
    on = (!e || atoi(e) != 0) ? 1 : 0;
  }
  return on == 1;
}

void tc_choose_pack_fmt(const DnRowsSrc& src, DnLayer* layers, int n_layers, int passes) {
  int fmt = (hybrid_enabled() && tc_chain3_supported(src, layers, n_layers) == DN_OK) ? 1 : 0;
  if (passes == DN_PASSES_BF16 && tc_chain16_supported(src, layers, n_layers) == DN_OK) fmt = 2;
  for (int l = 0; l < n_layers; ++l) layers[l].pack_fmt = fmt;
}

int64_t tc_chain_ws_bytes(const DnLayer* layers, int n_layers) {
  int64_t b = 0;
  for (int l = 0; l < n_layers; ++l) b += ((int64_t)layers[l].K * layers[l].N * 2 * 4 + 255) / 256 * 256;
  return b;
}

int tc_pack_layers(DnLayer* layers, int n_layers, void* ws, int64_t ws_bytes, cudaStream_t st) {
  return tc_pack_layers_spectral(layers, n_layers, ws, ws_bytes, nullptr, 0, nullptr, nullptr, 0, st);
}

int tc_pack_layers_spectral(DnLayer* layers, int n_layers, void* ws, int64_t ws_bytes, const float* partial, int P,
                            const float* evals, float* time, int clamp_writeback, cudaStream_t st) {
  if (n_layers < 1 || n_layers > DN_MAX_LAYERS) return DN_ERR_INVALID_ARGUMENT;
  if (tc_chain_ws_bytes(layers, n_layers) > ws_bytes || !ws) return DN_ERR_WORKSPACE;
  PackJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  jobs.sp_partial = partial; jobs.sp_P = P; jobs.sp_evals = evals; jobs.sp_time = time; jobs.sp_clamp = clamp_writeback;
  jobs.n = n_layers;
  jobs.kc = KC;
  char* wp = static_cast<char*>(ws);
  int blocks = 0;
  for (int l = 0; l < n_layers; ++l) {
    DnLayer& L = layers[l];
    PackJob& J = jobs.j[l];
    J.W = L.W; J.W2 = L.W2; J.n_split = L.n_split; J.ldw = L.ldw; J.w_trans = L.w_trans; J.K = L.K; J.N = L.N;
    J.fmt = L.pack_fmt;
    J.rot_C = L.rot_C; J.rot_ch0 = L.rot_ch0;
    J.dst = reinterpret_cast<float*>(wp);
    J.blk0 = blocks;
    blocks += (l == 0 && partial) ? (L.K * L.N + 31) / 32 : (L.K * L.N + 255) / 256;
    L.prepacked = J.dst;
    wp += ((int64_t)L.K * L.N * 2 * 4 + 255) / 256 * 256;
  }
  pack_weights_kernel<<<blocks, 256, 0, st>>>(jobs);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int tc_pack_spectral_batched(DnLayer* layer0, int n_meshes, void* ws, int64_t ws_bytes, const float* partial,
                             const int32_t* mesh_cta_begin, const float* evals, float* time, int clamp_writeback,
                             const int32_t* tile_mesh, cudaStream_t st, float* x_spec_out) {
  if (!layer0 || n_meshes < 1 || !ws || !partial || !mesh_cta_begin || !evals || !time || !tile_mesh)
    return DN_ERR_INVALID_ARGUMENT;
  const int64_t per = tc_chain_ws_bytes(layer0, 1);
  if (per * n_meshes > ws_bytes) return DN_ERR_WORKSPACE;
  const int K = layer0->K, N = layer0->N;
  dim3 grid((unsigned)((K * N + 31) / 32), (unsigned)n_meshes);
  spectral_pack_batched_kernel<<<grid, 256, 0, st>>>(partial, mesh_cta_begin, evals, time, K, N, layer0->pack_fmt, KC,
                                                     static_cast<float*>(ws), per / 4, clamp_writeback, x_spec_out);
  DN_LAUNCH_CHECK();
  layer0->prepacked = static_cast<float*>(ws);
  layer0->tile_group = tile_mesh;
  layer0->group_stride = per / 4;
  return DN_OK;
}

int64_t tc_spectral_bwd_batched_scratch_floats(int n_meshes, int K, int N) {
  return (int64_t)n_meshes * ((K + DN_SPEC_BWD_KROWS - 1) / DN_SPEC_BWD_KROWS) * N;
}

int tc_spectral_bwd_batched(DnLayer* layer0, int n_meshes, void* ws, int64_t ws_bytes, const float* partial,
                            const int32_t* mesh_cta_begin, const float* evals, const float* time, const float* x_spec,
                            float* dt_scratch, float* grad_time, const int32_t* tile_mesh, cudaStream_t st) {
  if (!layer0 || n_meshes < 1 || !ws || !partial || !mesh_cta_begin || !evals || !time || !x_spec || !dt_scratch ||
      !grad_time || !tile_mesh)
    return DN_ERR_INVALID_ARGUMENT;
  const int64_t per = tc_chain_ws_bytes(layer0, 1);
  if (per * n_meshes > ws_bytes) return DN_ERR_WORKSPACE;
  const int K = layer0->K, N = layer0->N;
  const int kgroups = (K + DN_SPEC_BWD_KROWS - 1) / DN_SPEC_BWD_KROWS;
  dim3 grid((unsigned)((N + 31) / 32), (unsigned)kgroups, (unsigned)n_meshes);
  spectral_bwd_pack_batched_kernel<<<grid, 256, 0, st>>>(partial, mesh_cta_begin, evals, time, x_spec, K, N,
                                                         layer0->pack_fmt, KC, static_cast<float*>(ws), per / 4, dt_scratch);
  DN_LAUNCH_CHECK();
  grad_time_reduce_kernel<<<(N + 31) / 32, 1024, 0, st>>>(dt_scratch, n_meshes * kgroups, N, grad_time);
  DN_LAUNCH_CHECK();
  layer0->prepacked = static_cast<float*>(ws);
  layer0->tile_group = tile_mesh;
  layer0->group_stride = per / 4;
  return DN_OK;
}

int tc_grouped_chain_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int passes) {
  if (passes == DN_PASSES_BF16 && tc_chain16_supported(src, layers, n_layers) == DN_OK) return DN_OK;
  return tc_chain3_supported(src, layers, n_layers);
}

int tc_rows_chain(const DnRowsSrc& src, const DnLayer* layers_in, int n_layers, int64_t V, int passes, void* ws,
                  int64_t ws_bytes, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  DevState* dv = cur_dev_state();
  if (!dv || dv->ok != 1) return DN_ERR_NOT_SM100;
  DnLayer layers[DN_MAX_LAYERS];
  bool packed = true;
  for (int l = 0; l < n_layers; ++l) {
    layers[l] = layers_in[l];
    packed = packed && layers[l].prepacked != nullptr;
  }
  if (!packed) {
    tc_choose_pack_fmt(src, layers, n_layers, passes);
    int rc = tc_pack_layers(layers, n_layers, ws, ws_bytes, st);
    if (rc) return rc;
  }
  if (passes == DN_PASSES_BF16) {
    // bf16 engine: the SS bf16 chain when the shapes fit it (weights packed as bf16), single-pass TF32 otherwise
    if (layers[0].pack_fmt == 2) return tc_rows_chain16(src, layers, n_layers, V, dv->sms, st);
    passes = 1;
  }
  // default: the TMA-fed kernel of dn_chain.cu; shapes outside its envelope run the round-1 kernels below
  if (tc_chain3_supported(src, layers, n_layers) == DN_OK) {
    const int rc = tc_rows_chain3(src, layers, n_layers, V, passes, dv->sms, take_trace_ptr(), st);
    if (rc != DN_ERR_UNSUPPORTED) return rc;
  }
  if (layers[0].tile_group) return DN_ERR_UNSUPPORTED;              // per-mesh layer-0 weights: chain3 / chain16 only
  for (int l = 0; l < n_layers; ++l)
    if (layers[l].pack_fmt != 0) return DN_ERR_INVALID_ARGUMENT;     // the round-1 kernels read the 16-wide chunk layout
  if (tc_rows_chain_legacy_supported(src, layers, n_layers) != DN_OK) return DN_ERR_UNSUPPORTED;
  TcChainParams p;
  memset(&p, 0, sizeof(p));
  p.src = src;
  p.n_layers = n_layers;
  p.passes = passes;
  p.V = V;
  p.trace = g_trace_ptr;
  p.nmax = 128;
  for (int l = 0; l < n_layers; ++l)
    if (layers[l].N > 128) p.nmax = 256;
  // TMEM plan of the TMEM-A kernel
  p.acc_col[0] = 0; p.acc_col[1] = 128; p.nbuf = 2; p.a_col0 = 256; p.nsa = 8;
  if (p.nmax == 256 && n_layers == 1) { p.acc_col[1] = 0; p.nbuf = 1; }
  if (p.nmax == 256 && n_layers == 2) { p.a_col0 = 384; p.nsa = 4; }   // [0,128) | [128,384) | ring [384,512)
  {
    // measured (V=200k): role specialisation wins on the 2-layer from_basis+[P|Q] chain (196 -> 167 us: few
    // layer-0 chunks, heavy epilogues) and loses on the MiniMLP (270 -> 280 us: 24 layer-0 chunks per tile)
    static int split_env = -2;
    if (split_env == -2) {
      const char* e = getenv("DN_TC_SPLIT");
      split_env = e ? atoi(e) : -1;
    }
    p.ts_split = split_env >= 0 ? split_env : (n_layers == 2 ? 1 : 0);
  }
  for (int l = 0; l < n_layers; ++l) {
    const DnLayer& L = layers[l];
    TcLayer& T = p.layer[l];
    T.wpack = L.prepacked; T.bias = L.bias; T.residual = L.residual; T.ld_res = L.ld_res; T.row_scale = L.row_scale;
    T.out = L.out; T.ld_out = L.ld_out; T.K = L.K; T.N = L.N; T.relu = L.relu;
  }
  const int64_t ntiles = (V + TILE_M - 1) / TILE_M;
  static int use_ts = -1;
  if (use_ts < 0) {
    const char* e = getenv("DN_TC_TS");
    use_ts = e ? atoi(e) : 2;   // 0: never, 1: always, 2 (default): for chained layers
  }
  if (use_ts == 1 || (use_ts == 2 && n_layers > 1)) {   // activations in TMEM (A operand read from tensor memory), one CTA per SM
    const int grid1 = (int)(ntiles < dv->sms ? ntiles : dv->sms);
    rows_chain_ts_kernel<<<grid1, TS_THREADS, TS_SMEM, st>>>(p);
    DN_LAUNCH_CHECK();
    return DN_OK;
  }
  const int grid = (int)(ntiles < 2 * dv->sms ? ntiles : 2 * dv->sms);
  rows_chain_kernel<<<grid, CHAIN_THREADS, CHAIN_SMEM, st>>>(p);
  DN_LAUNCH_CHECK();
  return DN_OK;
}

int tc_to_basis_supported(int K, int C) {
  if (K % 4 || K < 4 || K > 128) return DN_ERR_UNSUPPORTED;
  if (C % 16 || C < 16 || C > 128) return DN_ERR_UNSUPPORTED;
  return DN_OK;
}

int tc_to_basis_partial(const float* values, const float* basis, const float* massvec, int64_t V, int K, int C,
                        float* partial, int* P_out, int passes, cudaStream_t st, int64_t ld_values, int64_t ldp,
                        const int32_t* cta_rows, int n_ctas) {
  DevState* dv = cur_dev_state();
  if (!dv || dv->ok != 1) return DN_ERR_NOT_SM100;
  if (ld_values <= 0) ld_values = C;
  if (ldp <= 0) ldp = C;
  if ((reinterpret_cast<uintptr_t>(values) & 15) || (reinterpret_cast<uintptr_t>(basis) & 15) || (ld_values % 4) ||
      (ldp % 4) || (reinterpret_cast<uintptr_t>(partial) & 15))
    return DN_ERR_UNSUPPORTED;
  TcToBasisParams p;
  p.values = values; p.basis = basis; p.mass = massvec; p.partial = partial;
  p.ld_values = ld_values; p.ldp = ldp; p.cta_rows = cta_rows;
  if (cta_rows) {                       // batch of meshes: the caller planned the CTAs (dn_mesh_batch_plan)
    if (n_ctas < 1) return DN_ERR_INVALID_ARGUMENT;
    p.V = V; p.K = K; p.C = C; p.passes = (passes == 3) ? 3 : 1; p.chunks_per_cta = 0;
    to_basis_kernel<<<n_ctas, TB_THREADS, TB_SMEM, st>>>(p);
    DN_LAUNCH_CHECK();
    *P_out = n_ctas;
    return DN_OK;
  }
  p.V = V; p.K = K; p.C = C; p.passes = (passes == 3) ? 3 : 1;
  const int64_t total_chunks = (V + KC - 1) / KC;
  int grid = dv->sms;
  if (total_chunks < grid) grid = (int)(total_chunks > 0 ? total_chunks : 1);
  p.chunks_per_cta = (total_chunks + grid - 1) / grid;
  if (p.chunks_per_cta < 1) p.chunks_per_cta = 1;
  grid = (int)((total_chunks + p.chunks_per_cta - 1) / p.chunks_per_cta);
  if (grid < 1) grid = 1;
  to_basis_kernel<<<grid, TB_THREADS, TB_SMEM, st>>>(p);
  DN_LAUNCH_CHECK();
  *P_out = grid;
  return DN_OK;
}
