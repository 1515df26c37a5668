// TMA-fed fused affine chain over 128-vertex row tiles (sm_100a) -- the default tensor-core kernel for the
// dense layers of the DiffusionNetBlock path:
//     from_basis (+ the commuted complex-linear [P|Q])                 reference layers.py:64-67, 117-126
//     cat(x_in, x_diffuse, features) -> MiniMLP -> + x_in              reference layers.py:133-164, 229-239
//
// One persistent CTA per SM, 16 warps, every role fed by an mbarrier ring:
//   warp 0      weight producer: one bulk copy (cp.async.bulk) per 32-wide K-stage of pre-split weights
//               ([tf32 hi | bf16 (hi ; lo)], pack format 1)
//   warp 1      row-box producer: layer-0 operands as 128-row x 32-column fp32 boxes through TMA tensor maps
//               (SWIZZLE_128B), four slots
//   warp 2      MMA issuer, A operand from TENSOR MEMORY, B from shared memory: per 32-wide stage four
//               tcgen05.mma.kind::tf32 (hi*hi) and, fp32-grade, four kind::f16 bf16 MMAs for the correction terms, then
//               ONE tcgen05.commit that releases the TMEM operand stage and the weight stage together
//   warp 3      allocates / frees TMEM
//   warps 4-11  two operand warpgroups.  Stage c of every layer belongs to warpgroup c & 1 (so each ring slot has a
//               single in-order producer -- the mbarrier parity protocol needs that): layer-0 stages are read back
//               from the row box with conflict-free swizzled LDS.128, split x = hi + lo and written to the TMEM operand
//               ring with tcgen05.st; stages of a chained layer come from the previous accumulator
//               (tcgen05.ld -> bias / ReLU -> split -> tcgen05.st), never touching shared or global memory
//   warps 12-15 output warpgroup: every layer that has an HBM output: accumulator -> bias / ReLU / row scale
//               (+ residual, fetched by TMA into the staging slice) -> swizzled staging slice -> TMA store.  Each warp
//               owns the 32-row slices of the staging buffers for its TMEM lane quarter, issues its own TMA loads and
//               stores and tracks them with its own barriers / bulk groups: no cross-warp hand-off on the output path.
// Because the output warpgroup is separate, the operand warpgroups run straight from the last chained epilogue of a
// tile into the conversions of the next tile, and the MMA warp from the last layer of one tile into layer 0 of the
// next (accumulators ping-pong in TMEM).
//
// TMEM (512 columns): all N <= 128: accumulators [0,128) [128,256) ping-pong, operand ring [256,512) = 4 stages of
// (hi32 | lo32);  two-layer chain with N1 = 256 (from_basis -> [P|Q]): [0,128) | [128,384), ring [384,512) = 2 stages;
// single layer with N = 256: [0,256), ring [256,384) = 2 stages.
// Shared memory (224 KiB + barriers): row boxes 4 x 16 KiB | output staging 2 x 16 KiB | weight ring 128 KiB
// (4 x 32 KiB, or 2 x 64 KiB when a layer is 256 wide).
//
// Envelope: every K % 64 == 0, every N % 32 == 0, N <= 256 (see tc_chain3_supported); everything else runs the
// round-1 kernels in dn_tc.cu.
#include "dn_internal.h"
#include "dn_tc_ptx.cuh"
#include <cuda.h>
#include <string.h>

namespace {

using namespace tc;

constexpr int C3_THREADS = 512;
constexpr int C3_KS = 32;                       // k-columns per pipeline stage
constexpr int C3_TILE = 128;                    // rows per tile == UMMA M
constexpr int C3_RAW = C3_TILE * C3_KS * 4;     // 16 KiB row box
// row-box slots + output staging buffers share 6 x 16 KiB: 4 + 2.  (2 + 4 was measured on the output-heavy
// from_basis -> [P|Q] chain -- four layer-0 stages, 192 KiB of output per tile -- and was SLOWER, 124 vs 108 us: the
// extra staging traffic competes with the tensor core for shared-memory bandwidth.)
constexpr int C3_IO_BUFS = 6;
constexpr int C3_RAW_SHIFT = 2;                 // row-box slots = 1 << C3_RAW_SHIFT
constexpr int C3_RAW_SLOTS = 1 << C3_RAW_SHIFT;
constexpr int C3_WBYTES = 131072;               // weight ring
constexpr int C3_OFF_W = C3_IO_BUFS * C3_RAW;
constexpr int C3_OFF_BAR = C3_OFF_W + C3_WBYTES;
constexpr int C3_SMEM = C3_OFF_BAR + 512 /*barriers*/;

struct C3Layer {
  const float* wpack;      // tc_pack_layers layout, pack format 1 (32-wide stages of [tf32 hi | bf16 (hi ; lo)])
  const float* bias;       // [N] or null
  const float* row_scale;  // [V] or null (last layer only)
  int K, N, relu;
  int has_out;
  int has_res;             // 0: none | 1: + residual (layers.py:239) | 2: * (aux > 0): backward of ReLU, aux = the
                           //    forward activation (last layer only; the tensor is fetched through maps.res)
                           // 3: complex inner product + tanh (layers.py:128-130): accumulator = [Bre | Bim], N/2 columns
  int gy_col;              //    each; gX / gY boxes come through maps.res at columns c and gy_col + c; output N/2 wide
};

struct C3Params {
  C3Layer layer[DN_MAX_LAYERS];
  int n_layers, nsrc;
  int passes;      // 1: one TF32 MMA per product | 2: TF32 hi*hi + bf16 corrections
  int src_width[DN_MAX_SRC];
  int nbuf;        // accumulator buffers (2: ping-pong, column 128 * (g & 1); 1: column 0)
  int ring_col;    // first TMEM column of the operand ring
  int ns_shift;    // log2(ring depth): 2 -> 4 stages (32 KiB weight slots), 1 -> 2 stages (64 KiB weight slots)
  // linear head behind the LAST layer (DnLayer::head_*): its N-wide output row is consumed in registers, not stored
  const float* head_w;
  const float* head_b;
  float* head_out;
  int64_t ld_head_out;
  int head_n;
  int nio;         // 16 KiB row-box + staging buffers in front of the weight ring: 6 (weight ring 128 KiB) or 8 (96 KiB);
                   //   output staging buffers = nio - C3_RAW_SLOTS
  int64_t V;
  long long* trace;   // optional (tools/trace_chain3.py): per-warp (event, clock64) pairs of CTA 0
  const int32_t* tile_group;   // optional (mesh batches): layer 0 of tile t streams the packed matrix number tile_group[t]
  int64_t group_stride;        //   (floats between the per-mesh matrices)
};

struct C3Maps {
  CUtensorMap src[DN_MAX_SRC];      // 128-row x 32-column load boxes over the layer-0 sources
  CUtensorMap out[DN_MAX_LAYERS];   // 32-row x 32-column store boxes over each layer's output
  CUtensorMap res;                  // 32-row x 32-column load boxes over the last layer's residual
};

__device__ __forceinline__ void tma_box_load(uint32_t dst_smem, const CUtensorMap* tmap, int col, int row, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst_smem),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(col), "r"(row), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_box_store(const CUtensorMap* tmap, int col, int row, uint32_t src_smem) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(
                   reinterpret_cast<uint64_t>(tmap)),
               "r"(col), "r"(row), "r"(src_smem)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ float4 lds128(uint32_t a) {
  float4 r;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(a));
  return r;
}
__device__ __forceinline__ void sts128(uint32_t a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}

#define C3_TRACE_MAX 2048
#define C3_TRACE(ev)                                                                   \
  do {                                                                                 \
    if (p.trace && blockIdx.x == 0 && lane == 0 && tr_n < C3_TRACE_MAX) {              \
      p.trace[((int64_t)warp * C3_TRACE_MAX + tr_n) * 2] = (ev);                       \
      p.trace[((int64_t)warp * C3_TRACE_MAX + tr_n) * 2 + 1] = clock64();              \
      ++tr_n;                                                                          \
    }                                                                                  \
  } while (0)

template <bool HEAD>     // HEAD: the fused linear head path exists (its accumulators would cost the common path registers)
__global__ void __launch_bounds__(C3_THREADS, 1)
rows_chain3_kernel(const __grid_constant__ C3Params p, const __grid_constant__ C3Maps maps) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t smem0 = smem_u32(smem);
  if (smem0 & 1023u) __trap();                                          // SWIZZLE_128B boxes need 1024 B alignment
  const uint32_t nr_sh = C3_RAW_SHIFT, nr_mask = C3_RAW_SLOTS - 1;
  const uint32_t nout = (uint32_t)p.nio - C3_RAW_SLOTS, nout_mask = nout - 1u;        // 2 or 4
  const uint32_t raw_u = smem0, out_u = smem0 + (uint32_t)C3_RAW * C3_RAW_SLOTS, w_u = smem0 + (uint32_t)p.nio * C3_RAW;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C3_OFF_BAR);

  // bars: raw_full[4] raw_empty[4] full[4] ab_empty[4] dm_full[2] do_full[2] dm_empty[2] do_empty[2] res[4 warps][2] done
  //   full[s]     : operand stage s AND weight stage s are ready (4 operand-warp arrivals + the weight producer's
  //                 arrive.expect_tx): the MMA warp waits once per stage
  //   ab_empty[s] : one tcgen05.commit frees both
  //   dm_full / do_full [buf]: accumulator complete, for its chained-epilogue readers / for its output readers.  Two
  //                 barriers because each waiter must observe EVERY phase of a barrier it waits on (a parity wait
  //                 that skips a phase aliases): operand warps only follow layers that feed another layer, the output
  //                 warps only layers that have an HBM output.
  const uint32_t raw_full = smem_u32(bars), raw_empty = smem_u32(bars + 4);
  const uint32_t full = smem_u32(bars + 8), ab_empty = smem_u32(bars + 12);
  const uint32_t dm_full = smem_u32(bars + 16), do_full = smem_u32(bars + 18);
  const uint32_t dm_empty = smem_u32(bars + 20), do_empty = smem_u32(bars + 22);
  const uint32_t res_bar = smem_u32(bars + 24), done_bar = smem_u32(bars + 40);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 42);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int tr_n = 0;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) {
      mbar_init(raw_full + 8 * i, 1); mbar_init(raw_empty + 8 * i, 4);
      mbar_init(full + 8 * i, 5);     mbar_init(ab_empty + 8 * i, 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(dm_full + 8 * i, 1);  mbar_init(do_full + 8 * i, 1);
      mbar_init(dm_empty + 8 * i, 8); mbar_init(do_empty + 8 * i, 4);
    }
    for (int i = 0; i < 16; ++i) mbar_init(res_bar + 8 * i, 1);
    mbar_init(done_bar, 1);
    fence_barrier_init();
  }
  if (warp == 3) tmem_alloc<512>(smem_u32(tmem_slot));
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.nsrc; ++s) prefetch_tmap(&maps.src[s]);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int L = p.n_layers;
  const int64_t ntiles = (p.V + C3_TILE - 1) / C3_TILE;
  const int nst0 = p.layer[0].K / C3_KS;
  const uint32_t ns_sh = (uint32_t)p.ns_shift, ns_mask = (1u << ns_sh) - 1u;
  const uint32_t w_slot = (((uint32_t)C3_OFF_BAR - (uint32_t)p.nio * C3_RAW) >> ns_sh) & ~1023u;   // 32 / 64 KiB (nio 6), 48 KiB (nio 8)
  const bool two = p.nbuf == 2;

  if (warp == 0) {
    // ===================== weight producer =====================
    uint32_t i = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int l = 0; l < L; ++l) {
        const int N = p.layer[l].N, nst = p.layer[l].K / C3_KS;
        const uint32_t bytes = (uint32_t)N * 256u;              // two packed 16-wide chunks: hi | lo | hi | lo
        const float* wsrc = p.layer[l].wpack;
        if (l == 0 && p.tile_group) wsrc += (int64_t)__ldg(p.tile_group + tile) * p.group_stride;
        for (int c = 0; c < nst; ++c, ++i) {
          const uint32_t s = i & ns_mask;
          C3_TRACE(40);
          mbar_wait(ab_empty + 8 * s, ((i >> ns_sh) & 1) ^ 1);
          C3_TRACE(41);
          if (elect_one()) {
            mbar_arrive_expect_tx(full + 8 * s, bytes);
            tma_bulk_g2s(w_u + s * w_slot, wsrc + (int64_t)c * N * 64, bytes, full + 8 * s);
          }
          __syncwarp();
        }
      }
  } else if (warp == 1) {
    // ===================== row-box producer (layer-0 operands) =====================
    uint32_t r = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      int s = 0, k0 = 0;
      for (int c = 0; c < nst0; ++c, ++r) {
        const uint32_t sl = r & nr_mask;
        C3_TRACE(50);
        mbar_wait(raw_empty + 8 * sl, ((r >> nr_sh) & 1) ^ 1);
        C3_TRACE(51);
        if (elect_one()) {
          mbar_arrive_expect_tx(raw_full + 8 * sl, C3_RAW);
          tma_box_load(raw_u + sl * C3_RAW, &maps.src[s], k0, (int)(tile * C3_TILE), raw_full + 8 * sl);
        }
        __syncwarp();
        k0 += C3_KS;
        if (k0 == p.src_width[s]) { k0 = 0; ++s; }
      }
    }
  } else if (warp == 2) {
    // ===================== MMA issuer =====================
    const uint32_t w_u4 = w_u >> 4;
    uint32_t i = 0, g = 0;
    uint32_t cm0 = 0, cm1 = 0, co0 = 0, co1 = 0;      // completed main / output drains announced per buffer
    uint32_t pend = 0;                                // bit 0/1: main drain pending on buffer 0/1, bit 2/3: output drain
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      for (int l = 0; l < L; ++l, ++g) {
        const int N = p.layer[l].N, nst = p.layer[l].K / C3_KS;
        const uint32_t idesc = make_idesc_tf32(C3_TILE, N), idesc16 = make_idesc_bf16(C3_TILE, N);
        const uint32_t buf = two ? (g & 1u) : 0u;
        const uint32_t d_tmem = tmem_base + buf * 128u;
        const uint32_t b_lbo = (uint32_t)N * 16u;
        const uint64_t tmplB = make_desc(0, b_lbo, 128);
        const uint32_t kg2 = (2u * b_lbo) >> 4;           // k-group stride of both stage images (N * 16 B)
        // the previous user of this accumulator must have been drained by everyone who reads it
        C3_TRACE(23);
        if (pend & (1u << buf)) {
          mbar_wait(dm_empty + 8 * buf, ((buf ? cm1 : cm0) - 1u) & 1u);
          pend &= ~(1u << buf);
        }
        if (pend & (4u << buf)) {
          mbar_wait(do_empty + 8 * buf, ((buf ? co1 : co0) - 1u) & 1u);
          pend &= ~(4u << buf);
        }
        tc_fence_after();
        C3_TRACE(24);
        // Stages are handed over in PAIRS when the ring has four slots: the fixed cost of a hand-off in this warp (barrier
        // poll, fence, elect, descriptor setup, commits: ~450 cycles during which the tensor pipe drains -- the MMA queue
        // is shallow, `tcgen05.mma` issue blocks for about the execution time) is then paid once per 16 MMAs instead of
        // once per 8, while the operand warps fill the other two slots.  (A 128x128x8 MMA retires in 64 cycles when MMAs
        // are issued back to back, tools/ubench/ubench3.cu: 8 per stage = 512 cycles against ~1100 measured per stage.)
        const int step = (ns_sh == 2) ? 2 : 1;
        for (int c = 0; c < nst; c += step, i += (uint32_t)step) {
          C3_TRACE(20);
          for (int h = 0; h < step; ++h) mbar_wait(full + 8 * ((i + (uint32_t)h) & ns_mask), ((i + (uint32_t)h) >> ns_sh) & 1u);
          C3_TRACE(21);
          tc_fence_after();
          if (elect_one()) {
            for (int h = 0; h < step; ++h) {
              const uint32_t s = (i + (uint32_t)h) & ns_mask;
              const int cc = c + h;
              const uint32_t a0 = tmem_base + (uint32_t)p.ring_col + s * 64u;
              const uint64_t dbs = tmplB + (w_u4 + s * (w_slot >> 4));
              // stage = [tf32 hi image | bf16 (hi ; lo) image].  Four TF32 MMAs (K = 8) form hi*hi; with two passes four
              // bf16 MMAs (K = 16) add the corrections [x_lo | x_hi] . [W_hi ; W_lo] -- 8 instructions and 32 KiB of
              // shared-memory operand reads per stage where 3xTF32 needs 12 and 48 KiB, same fp32-grade result
#pragma unroll
              for (int ks = 0; ks < 4; ++ks)
                mma_tf32_ts(d_tmem, a0 + ks * 8, dbs + (uint32_t)ks * kg2, idesc, (cc | ks) ? 1u : 0u);
              if (p.passes == 2) {
                const uint64_t db16 = dbs + (((uint32_t)N * 128u) >> 4);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                  mma_f16_ts(d_tmem, a0 + 32 + j * 8, db16 + (uint32_t)j * kg2, idesc16, 1u);
              }
              mma_commit(ab_empty + 8 * s);           // frees TMEM operand stage s and weight stage s
            }
            if (c + step == nst) {
              if (l + 1 < L) mma_commit(dm_full + 8 * buf);
              if (p.layer[l].has_out) mma_commit(do_full + 8 * buf);
            }
          }
          __syncwarp();
          C3_TRACE(22);
        }
        if (l + 1 < L) { pend |= (1u << buf); if (buf) ++cm1; else ++cm0; }
        if (p.layer[l].has_out) { pend |= (4u << buf); if (buf) ++co1; else ++co0; }
      }
    // never leave the CTA with tensor-core work in flight (TMEM is freed and the barriers die at exit)
    if (elect_one()) mma_commit(done_bar);
    __syncwarp();
    mbar_wait(done_bar, 0);
  } else if (warp >= 4 && warp < 12) {
    // ===================== operand warpgroups: layer-0 conversion + chained epilogues =====================
    const uint32_t wg = (uint32_t)(warp - 4) >> 2;      // owns stages with (c & 1) == wg
    const int quarter = warp & 3;                       // TMEM lane quarter: this lane owns tile row 32*quarter + lane
    const int trow = 32 * quarter + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(32 * quarter) << 16);
    const uint32_t swz = (uint32_t)(trow & 7);

    // x[32] -> (hi32 | lo32) in ring stage (i mod depth), then hand the stage to the MMA warp
    auto put_stage = [&](uint32_t i, const float* x) {
      const uint32_t s = i & ns_mask;
      C3_TRACE(3);
      mbar_wait(ab_empty + 8 * s, ((i >> ns_sh) & 1u) ^ 1u);
      C3_TRACE(4);
      tc_fence_after();
      const uint32_t ta = lane_base + (uint32_t)p.ring_col + s * 64u;
      if (p.passes == 2) {
        // columns [0,32): tf32 hi | [32,48): bf16x2 pairs of lo = x - hi | [48,64): bf16x2 pairs of hi
        float plo[16], phi[16];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) split_tf32_fast(x[16 * h + j], hi[j], lo[j]);
          tmem_st16(ta + 16 * h, hi);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            plo[8 * h + j] = __uint_as_float(pack_bf16x2(lo[2 * j], lo[2 * j + 1]));
            phi[8 * h + j] = __uint_as_float(pack_bf16x2(hi[2 * j], hi[2 * j + 1]));
          }
        }
        tmem_st16(ta + 32, plo);
        tmem_st16(ta + 48, phi);
      } else {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          float hi[16], lo[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) split_tf32_fast(x[16 * h + j], hi[j], lo[j]);
          tmem_st16(ta + 16 * h, hi);
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(full + 8 * s);
      C3_TRACE(5);
    };

    uint32_t t_seq = 0;
    uint32_t um0 = 0, um1 = 0;                          // chained-epilogue uses of accumulator buffer 0 / 1 so far
    int S = 0;
    for (int l = 0; l < L; ++l) S += p.layer[l].K / C3_KS;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++t_seq) {
      const uint32_t i_base = t_seq * (uint32_t)S, r_base = t_seq * (uint32_t)nst0;
      // ---- layer 0: my stages of the row boxes -> TMEM
      for (int c = (int)wg; c < nst0; c += 2) {
        const uint32_t r = r_base + (uint32_t)c, sl = r & nr_mask;
        C3_TRACE(1);
        mbar_wait(raw_full + 8 * sl, (r >> nr_sh) & 1u);
        C3_TRACE(2);
        const uint32_t rowaddr = raw_u + sl * C3_RAW + (uint32_t)trow * 128u;
        float x[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 q = lds128(rowaddr + ((((uint32_t)j) ^ swz) << 4));
          x[4 * j] = q.x; x[4 * j + 1] = q.y; x[4 * j + 2] = q.z; x[4 * j + 3] = q.w;
        }
        // the slot release must not overtake the loads (LDS and mbarrier.arrive run in different pipes): really consume
        // one register of each 16-byte load first (consume_loaded)
        consume_loaded(((__float_as_uint(x[0]) ^ __float_as_uint(x[4])) ^ (__float_as_uint(x[8]) ^ __float_as_uint(x[12]))) ^
                       ((__float_as_uint(x[16]) ^ __float_as_uint(x[20])) ^ (__float_as_uint(x[24]) ^ __float_as_uint(x[28]))));
        __syncwarp();
        if (lane == 0) mbar_arrive(raw_empty + 8 * sl);
        put_stage(i_base + (uint32_t)c, x);
      }
      // ---- chained layers: accumulator l -> operand stages of layer l + 1
      uint32_t ib = i_base + (uint32_t)nst0;
      for (int l = 0; l + 1 < L; ++l) {
        const C3Layer& Lr = p.layer[l];
        const uint32_t g = t_seq * (uint32_t)L + (uint32_t)l;
        const uint32_t buf = two ? (g & 1u) : 0u;
        const int nco = Lr.N / C3_KS;
        C3_TRACE(10);
        mbar_wait(dm_full + 8 * buf, (buf ? um1 : um0) & 1u);
        C3_TRACE(11);
        if (buf) ++um1; else ++um0;
        tc_fence_after();
        const uint32_t d_lane = lane_base + buf * 128u;
        bool released = false;
        for (int c = (int)wg; c < nco; c += 2) {
          float v[32];
          // the chunk's 32 bias values: eight uniform-address (broadcast) 16-byte loads, in flight during the TMEM read
          // (a 32-step shuffle broadcast of per-lane values cost ~450 cycles on the critical path of every layer boundary)
          float4 b4[8];
          if (Lr.bias) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) b4[jj] = __ldg(reinterpret_cast<const float4*>(Lr.bias + c * C3_KS) + jj);
          }
          tmem_ld32(d_lane + (uint32_t)c * C3_KS, v);
          C3_TRACE(12);
          if (c + 2 >= nco) {                                    // my last read of this accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(dm_empty + 8 * buf);
            released = true;
          }
          if (Lr.bias) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              v[4 * jj] += b4[jj].x; v[4 * jj + 1] += b4[jj].y; v[4 * jj + 2] += b4[jj].z; v[4 * jj + 3] += b4[jj].w;
            }
          }
          if (Lr.relu) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          put_stage(ib + (uint32_t)c, v);
        }
        if (!released) {                                         // (a 32-wide layer gives warpgroup 1 nothing to read)
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(dm_empty + 8 * buf);
        }
        ib += (uint32_t)nco;
      }
    }
  } else if (warp >= 12) {
    // ===================== output warpgroup =====================
    const int quarter = warp & 3;
    const int trow = 32 * quarter + lane;
    const uint32_t lane_base = tmem_base + ((uint32_t)(32 * quarter) << 16);
    const uint32_t swz = (uint32_t)(lane & 7);                   // slices start on a 1024 B boundary: row-in-slice & 7
    const uint32_t my_res = res_bar + 8u * (uint32_t)(quarter * 4);
    uint32_t oc = 0;                 // output chunks issued so far (staging buffer = oc mod nout)
    uint32_t rcbits = 0;             // bit b: parity of the residual loads waited so far on staging buffer b
    uint32_t uo0 = 0, uo1 = 0;       // output uses of accumulator buffer 0 / 1 so far
    uint32_t t_seq = 0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++t_seq) {
      const int row0 = (int)(tile * C3_TILE) + 32 * quarter;
      const int64_t row = tile * C3_TILE + trow;
      for (int l = 0; l < L; ++l) {
        const C3Layer& Lr = p.layer[l];
        if (!Lr.has_out) continue;
        const uint32_t g = t_seq * (uint32_t)L + (uint32_t)l;
        const uint32_t buf = two ? (g & 1u) : 0u;
        const uint32_t use = buf ? uo1 : uo0;
        if (buf) ++uo1; else ++uo0;
        const int nco = Lr.N / C3_KS;
        const uint32_t d_lane = lane_base + buf * 128u;
        if (Lr.has_res == 3) {
          // feat = tanh(gX * Bre + gY * Bim): per 32-channel chunk two accumulator reads and two TMA boxes (gX into
          // this warp's slice of staging buffer 0, gY into buffer 1); the result overwrites slice 0 and is stored
          const int half = Lr.N >> 1, nch = half / C3_KS;
          const uint32_t slq = out_u + (uint32_t)quarter * 4096u;
          // with four staging buffers (nio == 8) every gX / gY box of the tile is requested before the accumulator is
          // awaited: the loads overlap the tile's MMAs instead of sitting between the accumulator and the store
          const bool pre = (int)nout >= 2 * nch;
          if (pre && lane == 0) {
            bulk_wait_read<0>();                                 // the previous tile's stores have left the slices
            for (int c = 0; c < nch; ++c) {
              mbar_arrive_expect_tx(my_res + 16 * c, 4096);
              tma_box_load(slq + (uint32_t)(2 * c) * C3_RAW, &maps.res, c * C3_KS, row0, my_res + 16 * c);
              mbar_arrive_expect_tx(my_res + 16 * c + 8, 4096);
              tma_box_load(slq + (uint32_t)(2 * c + 1) * C3_RAW, &maps.res, Lr.gy_col + c * C3_KS, row0, my_res + 16 * c + 8);
            }
          }
          __syncwarp();
          mbar_wait(do_full + 8 * buf, use & 1u);
          tc_fence_after();
          for (int c = 0; c < nch; ++c) {
            const int sb = pre ? 2 * c : 0;                      // staging buffers of this chunk: sb (gX, result), sb + 1 (gY)
            const uint32_t sl0 = slq + (uint32_t)sb * C3_RAW, sl1 = sl0 + C3_RAW;
            if (!pre) {
              if (lane == 0) {
                bulk_wait_read<0>();
                mbar_arrive_expect_tx(my_res, 4096);
                tma_box_load(sl0, &maps.res, c * C3_KS, row0, my_res);
                mbar_arrive_expect_tx(my_res + 8, 4096);
                tma_box_load(sl1, &maps.res, Lr.gy_col + c * C3_KS, row0, my_res + 8);
              }
              __syncwarp();
            }
            float re[32], im[32];
            tmem_ld32(d_lane + (uint32_t)c * C3_KS, re);
            tmem_ld32(d_lane + (uint32_t)(half + c * C3_KS), im);
            if (c + 1 == nch) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(do_empty + 8 * buf);
            }
            mbar_wait(my_res + 8 * sb, (rcbits >> sb) & 1u);
            mbar_wait(my_res + 8 * sb + 8, (rcbits >> (sb + 1)) & 1u);
            rcbits ^= (3u << sb);
            const uint32_t r0 = sl0 + (uint32_t)lane * 128u, r1 = sl1 + (uint32_t)lane * 128u;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              const uint32_t o = (((uint32_t)jj) ^ swz) << 4;
              const float4 gx = lds128(r0 + o), gy = lds128(r1 + o);
              sts128(r0 + o, dn_feat_tanh(fmaf(gx.x, re[4 * jj], gy.x * im[4 * jj])),
                     dn_feat_tanh(fmaf(gx.y, re[4 * jj + 1], gy.y * im[4 * jj + 1])),
                     dn_feat_tanh(fmaf(gx.z, re[4 * jj + 2], gy.z * im[4 * jj + 2])),
                     dn_feat_tanh(fmaf(gx.w, re[4 * jj + 3], gy.w * im[4 * jj + 3])));
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_box_store(&maps.out[l], c * C3_KS, row0, sl0);
              bulk_commit();
            }
            __syncwarp();
          }
          continue;
        }
        const bool res = Lr.has_res != 0;
        const float rs = (Lr.row_scale && row < p.V) ? __ldg(Lr.row_scale + row) : 1.f;
        const bool head = HEAD && p.head_w != nullptr && l + 1 == L;
        float ho[8];
        if (head) {
#pragma unroll
          for (int o = 0; o < 8; ++o) ho[o] = (o < p.head_n && p.head_b) ? __ldg(p.head_b + o) : 0.f;
        }
        C3_TRACE(30);
        if (!res) {
          mbar_wait(do_full + 8 * buf, use & 1u);
          tc_fence_after();
          C3_TRACE(31);
        }
        for (int c0 = 0; c0 < nco; c0 += (int)nout) {
          const int ng = (nco - c0) < (int)nout ? (nco - c0) : (int)nout;
          if (res) {
            // this group's residual slices: fetched by TMA into the staging slices the results will overwrite
            if (lane == 0) {
              bulk_wait_read<0>();                               // every earlier store has left its slice
              for (int j = 0; j < ng; ++j) {
                const uint32_t b = (oc + (uint32_t)j) & nout_mask;
                mbar_arrive_expect_tx(my_res + 8 * b, 4096);
                tma_box_load(out_u + b * C3_RAW + (uint32_t)quarter * 4096u, &maps.res, (c0 + j) * C3_KS, row0,
                             my_res + 8 * b);
              }
            }
            __syncwarp();
            if (c0 == 0) {
              mbar_wait(do_full + 8 * buf, use & 1u);
              tc_fence_after();
              C3_TRACE(31);
            }
          }
          for (int j = 0; j < ng; ++j, ++oc) {
            const int c = c0 + j;
            const uint32_t b = oc & nout_mask;
            const uint32_t slice = out_u + b * C3_RAW + (uint32_t)quarter * 4096u;
            if (!res) {
              if (lane == 0) {                                   // the store that last used this slice has read it
                if (nout == 4) bulk_wait_read<3>(); else bulk_wait_read<1>();
              }
              __syncwarp();
            }
            C3_TRACE(32);
            float v[32];
            float4 b4[8];                                        // bias of the chunk: broadcast loads under the TMEM read
            if (Lr.bias) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) b4[jj] = __ldg(reinterpret_cast<const float4*>(Lr.bias + c * C3_KS) + jj);
            }
            tmem_ld32(d_lane + (uint32_t)c * C3_KS, v);
            C3_TRACE(33);
            if (c + 1 == nco) {                                  // last read of this accumulator by this warp
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(do_empty + 8 * buf);
            }
            if (Lr.bias) {
#pragma unroll
              for (int jj = 0; jj < 8; ++jj) {
                v[4 * jj] += b4[jj].x; v[4 * jj + 1] += b4[jj].y; v[4 * jj + 2] += b4[jj].z; v[4 * jj + 3] += b4[jj].w;
              }
            }
            if (Lr.relu) {
#pragma unroll
              for (int jj = 0; jj < 32; ++jj) v[jj] = fmaxf(v[jj], 0.f);
            }
            if (Lr.row_scale) {
#pragma unroll
              for (int jj = 0; jj < 32; ++jj) v[jj] *= rs;
            }
            const uint32_t rowaddr = slice + (uint32_t)lane * 128u;
            if (res) {
              mbar_wait(my_res + 8 * b, (rcbits >> b) & 1u);
              C3_TRACE(34);
              rcbits ^= (1u << b);
              if (Lr.has_res == 1) {
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                  const float4 q = lds128(rowaddr + ((((uint32_t)jj) ^ swz) << 4));
                  v[4 * jj] += q.x; v[4 * jj + 1] += q.y; v[4 * jj + 2] += q.z; v[4 * jj + 3] += q.w;
                }
              } else {
#pragma unroll
                for (int jj = 0; jj < 8; ++jj) {
                  const float4 q = lds128(rowaddr + ((((uint32_t)jj) ^ swz) << 4));
                  v[4 * jj] = q.x > 0.f ? v[4 * jj] : 0.f;         v[4 * jj + 1] = q.y > 0.f ? v[4 * jj + 1] : 0.f;
                  v[4 * jj + 2] = q.z > 0.f ? v[4 * jj + 2] : 0.f; v[4 * jj + 3] = q.w > 0.f ? v[4 * jj + 3] : 0.f;
                }
              }
            }
            if (head) {
              // the fused linear head: this lane's row, 32 more input channels; the weights are uniform-address loads
#pragma unroll
              for (int o = 0; o < 8; ++o) {
                if (o < p.head_n) {
                  const float4* wr = reinterpret_cast<const float4*>(p.head_w + (int64_t)o * Lr.N + c * C3_KS);
                  float a = ho[o];
#pragma unroll
                  for (int jj = 0; jj < 8; ++jj) {
                    const float4 w = __ldg(wr + jj);
                    a = fmaf(w.x, v[4 * jj], a); a = fmaf(w.y, v[4 * jj + 1], a);
                    a = fmaf(w.z, v[4 * jj + 2], a); a = fmaf(w.w, v[4 * jj + 3], a);
                  }
                  ho[o] = a;
                }
              }
              if (res) {                                         // the residual slice was only read: it may be reloaded
                consume_loaded(__float_as_uint(ho[0]));
                __syncwarp();
              }
              C3_TRACE(35);
              continue;
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj)
              sts128(rowaddr + ((((uint32_t)jj) ^ swz) << 4), v[4 * jj], v[4 * jj + 1], v[4 * jj + 2], v[4 * jj + 3]);
            fence_proxy_async();                                 // generic-proxy writes -> visible to the TMA store
            __syncwarp();
            if (lane == 0) {
              tma_box_store(&maps.out[l], c * C3_KS, row0, slice);
              bulk_commit();
            }
            __syncwarp();
            C3_TRACE(35);
          }
        }
        if (head && row < p.V) {
          float* orow = p.head_out + row * p.ld_head_out;
#pragma unroll
          for (int o = 0; o < 8; ++o)
            if (o < p.head_n) orow[o] = ho[o];
        }
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // every store has completed
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 3) tmem_dealloc<512>(tmem_base);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*TmaEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
TmaEncodeFn tma_encode_fn() {
  static TmaEncodeFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<TmaEncodeFn>(f);
    else
      cudaGetLastError();
  }
  return fn;
}

// rows x width fp32 matrix (leading dimension ld) -> box_rows x 32-column boxes, SWIZZLE_128B; rows past V read as
// zeros and are not written
int make_box_map(CUtensorMap* m, const float* ptr, int width, int64_t ld, int64_t V, int box_rows) {
  const cuuint64_t dims[2] = {(cuuint64_t)width, (cuuint64_t)V};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
  const cuuint32_t box[2] = {(cuuint32_t)C3_KS, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = tma_encode_fn()(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box,
                                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : 1;
}

constexpr int kMaxDev = 64;
int g_attr_dev[kMaxDev];     // 0: not tried, 1: ok, -1: failed

}  // namespace

int tc_chain3_supported(const DnRowsSrc& src, const DnLayer* layers, int n_layers) {
  if (tma_encode_fn() == nullptr) return DN_ERR_UNSUPPORTED;
  if (n_layers < 1 || n_layers > DN_MAX_LAYERS) return DN_ERR_UNSUPPORTED;
  int k0 = 0;
  for (int s = 0; s < src.nsrc; ++s) {
    if (src.width[s] % C3_KS || src.ld[s] % 4 || (reinterpret_cast<uintptr_t>(src.ptr[s]) & 15)) return DN_ERR_UNSUPPORTED;
    k0 += src.width[s];
  }
  if (k0 != layers[0].K) return DN_ERR_UNSUPPORTED;
  int nmax = 0;
  for (int l = 0; l < n_layers; ++l) {
    const DnLayer& L = layers[l];
    const bool last = (l + 1 == n_layers);
    if (L.K % 64 || L.K < 64 || L.N % C3_KS || L.N < C3_KS || L.N > 256) return DN_ERR_UNSUPPORTED;
    if (L.emul) return DN_ERR_UNSUPPORTED;
    if (L.relu_mask_src && (!last || L.residual || (reinterpret_cast<uintptr_t>(L.relu_mask_src) & 15)))
      return DN_ERR_UNSUPPORTED;
    if (L.bias && (reinterpret_cast<uintptr_t>(L.bias) & 15)) return DN_ERR_UNSUPPORTED;
    if (!last && (L.residual || L.row_scale)) return DN_ERR_UNSUPPORTED;
    if (L.dots_src && (!last || L.residual || L.relu_mask_src || L.row_scale || L.bias || L.relu || (L.N % 64) || L.N > 128 ||
                       (L.ld_dots % 4) || (L.dots_gy_col % 4) || (reinterpret_cast<uintptr_t>(L.dots_src) & 15)))
      return DN_ERR_UNSUPPORTED;
    if (!last && L.N % 64) return DN_ERR_UNSUPPORTED;             // it is the next layer's K
    if (L.residual && (L.res_scale != 1.f || L.ld_res % 4 || (reinterpret_cast<uintptr_t>(L.residual) & 15)))
      return DN_ERR_UNSUPPORTED;
    if (L.out && (L.ld_out % 4 || (reinterpret_cast<uintptr_t>(L.out) & 15))) return DN_ERR_UNSUPPORTED;
    if (l > 0 && L.K != layers[l - 1].N) return DN_ERR_UNSUPPORTED;
    if (L.N > nmax) nmax = L.N;
  }
  {
    const DnLayer& Ll = layers[n_layers - 1];
    if (Ll.head_w) {
      if (!Ll.head_out || Ll.head_n < 1 || Ll.head_n > 8 || Ll.dots_src || Ll.relu_mask_src ||
          (reinterpret_cast<uintptr_t>(Ll.head_w) & 15))
        return DN_ERR_UNSUPPORTED;
    } else if (!Ll.out) {
      return DN_ERR_UNSUPPORTED;
    }
  }
  // TMEM plans: all N <= 128 | {N0 <= 128, N1 <= 256} | single layer N <= 256
  if (nmax > 128 && !(n_layers == 1 || (n_layers == 2 && layers[0].N <= 128))) return DN_ERR_UNSUPPORTED;
  return DN_OK;
}

int tc_rows_chain3(const DnRowsSrc& src, const DnLayer* layers, int n_layers, int64_t V, int passes, int sm_count,
                   long long* trace, cudaStream_t st) {
  if (V <= 0) return DN_OK;
  if (V >= (1ll << 31) - 256) return DN_ERR_UNSUPPORTED;
  int dev = 0;
  DN_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDev) return DN_ERR_UNSUPPORTED;
  if (g_attr_dev[dev] == 0) {                                      // function attributes are per device
    g_attr_dev[dev] =
        (cudaFuncSetAttribute(rows_chain3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C3_SMEM) == cudaSuccess &&
         cudaFuncSetAttribute(rows_chain3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C3_SMEM) == cudaSuccess) ? 1 : -1;
    if (g_attr_dev[dev] < 0) cudaGetLastError();
  }
  if (g_attr_dev[dev] < 0) return DN_ERR_UNSUPPORTED;

  C3Params p;
  C3Maps maps;
  memset(&p, 0, sizeof(p));
  memset(&maps, 0, sizeof(maps));
  p.n_layers = n_layers;
  for (int l = 0; l < n_layers; ++l)
    if (layers[l].pack_fmt != 1) return DN_ERR_INVALID_ARGUMENT;   // stage layout [tf32 hi | bf16 (hi ; lo)]
  p.passes = (passes == 3) ? 2 : 1;

  p.V = V;
  p.trace = trace;
  p.tile_group = layers[0].tile_group;
  p.group_stride = layers[0].group_stride;
  {
    const DnLayer& Ll = layers[n_layers - 1];
    p.head_w = Ll.head_w; p.head_b = Ll.head_b; p.head_out = Ll.head_out; p.ld_head_out = Ll.ld_head_out; p.head_n = Ll.head_n;
  }
  p.nsrc = src.nsrc;
  int nmax = 0;
  for (int s = 0; s < src.nsrc; ++s) {
    p.src_width[s] = src.width[s];
    if (make_box_map(&maps.src[s], src.ptr[s], src.width[s], src.ld[s], V, C3_TILE)) return DN_ERR_UNSUPPORTED;
  }
  for (int l = 0; l < n_layers; ++l) {
    const DnLayer& L = layers[l];
    C3Layer& T = p.layer[l];
    if (!L.prepacked) return DN_ERR_INVALID_ARGUMENT;
    T.wpack = L.prepacked; T.bias = L.bias; T.row_scale = L.row_scale; T.K = L.K; T.N = L.N; T.relu = L.relu;
    T.has_out = L.out != nullptr || (l + 1 == n_layers && L.head_w != nullptr);
    T.has_res = L.residual ? 1 : (L.relu_mask_src ? 2 : (L.dots_src ? 3 : 0));
    T.gy_col = L.dots_gy_col;
    if (L.dots_src) {     // output is N/2 wide; gX / gY boxes come from dots_src (any width >= gy_col + N/2)
      if (!L.out || make_box_map(&maps.out[l], L.out, L.N / 2, L.ld_out, V, 32)) return DN_ERR_UNSUPPORTED;
      if (make_box_map(&maps.res, L.dots_src, L.dots_gy_col + L.N / 2, L.ld_dots, V, 32)) return DN_ERR_UNSUPPORTED;
      if (L.N > nmax) nmax = L.N;
      continue;
    }
    if (L.out && make_box_map(&maps.out[l], L.out, L.N, L.ld_out, V, 32)) return DN_ERR_UNSUPPORTED;
    if (L.residual && make_box_map(&maps.res, L.residual, L.N, L.ld_res, V, 32)) return DN_ERR_UNSUPPORTED;
    if (L.relu_mask_src && make_box_map(&maps.res, L.relu_mask_src, L.N, L.N, V, 32)) return DN_ERR_UNSUPPORTED;
    if (L.N > nmax) nmax = L.N;
  }
  if (nmax <= 128) { p.nbuf = 2; p.ring_col = 256; p.ns_shift = 2; }
  else if (n_layers == 2) { p.nbuf = 2; p.ring_col = 384; p.ns_shift = 1; }
  else { p.nbuf = 1; p.ring_col = 256; p.ns_shift = 1; }
  p.nio = C3_IO_BUFS;
  if (n_layers == 1 && layers[0].dots_src && nmax <= 128) {
    // complex-dots layer: 4 row boxes + 4 staging buffers (all gX / gY boxes of a tile prefetched) + a 2-stage ring
    p.nio = 8; p.ns_shift = 1;
  }

  const int64_t ntiles = (V + C3_TILE - 1) / C3_TILE;
  const int grid = (int)(ntiles < sm_count ? ntiles : sm_count);
  if (p.head_w) rows_chain3_kernel<true><<<grid, C3_THREADS, C3_SMEM, st>>>(p, maps);
  else rows_chain3_kernel<false><<<grid, C3_THREADS, C3_SMEM, st>>>(p, maps);
  DN_LAUNCH_CHECK();
  return DN_OK;
}
