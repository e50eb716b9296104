// tc_gemm.cu — hand-written tcgen05 GEMM for the PPO policy/value MLPs (sm_100a).
//
//   C[M,N] = epilogue( A[M,K] · B[N,K]^T ),  A and B bf16 row-major (K contiguous), fp32 accumulate in TMEM.
//
// Replaces the cuBLAS sgemm + bias + tanh launches behind `nn.Linear`/`nn.Tanh` of the reference's
// `Agent` (ppo_continuous_action_isaacgym.py:127-164) and their autograd backward (:352).
// Persistent CTAs (two per SM) walk the 128 x BN output tiles (times K-splits):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D tiles (128B swizzle) into a 3-stage smem ring
//   warp 1      TMEM allocator + MMA issuer: one elected thread issues tcgen05.mma (M=128, N=BN, K=16)
//               into one of two TMEM accumulator buffers; tcgen05.commit releases smem stages and
//               signals the accumulator
//   warps 2-5   epilogue (one warp per TMEM lane quarter): tcgen05.ld 32 lanes x 32 columns, fused bias+tanh /
//               tanh-derivative / split-K fp32 atomics, vectorised global stores
// Every mbarrier wait is bounded (trap instead of hanging the GPU).
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <string>

#include "../../include/vss_b200.h"
#include "tc_common.cuh"

namespace tc {

constexpr int STAGES = 3;    // 3 x 32 KB: two CTAs per SM, so one CTA's epilogue overlaps the other's MMAs
constexpr int EPI_WARPS = 4;       // one warp per TMEM lane quarter (8 = two per quarter was measured: no gain, the kernel is operand-feed bound)
constexpr int THREADS = 64 + 32 * EPI_WARPS;

enum Epilogue : int {
  EPI_BIAS_TANH_BF16 = 0,  // out_bf16 = tanh(acc + bias[n])                       (forward hidden layer)
  EPI_DTANH_BF16 = 1,      // out_bf16 = acc * (1 - aux[m,n]^2), aux bf16           (dgrad fused with tanh')
  EPI_ATOMIC_F32 = 2,      // out_f32 += acc  (red.global.add.f32, split-K)         (wgrad)
  EPI_BIAS_F32 = 3,        // out_f32 = acc + bias[n]                               (plain linear)
};

struct GemmArgs {
  int M, N, K;             // problem; K multiple of 64, N multiple of BN
  int k_blocks_per_split;  // k-blocks (of 64) handled by one K-split
  int splits;              // number of K-splits (tiles = m_tiles * n_tiles * splits)
  int ws_stages;           // weight-stationary kernel: depth of the activation ring
  void* out;               // bf16 or f32, row-major [M, ldo]
  int ldo;
  const float* bias;       // [N] or null
  const __nv_bfloat16* aux;  // [M, ld_aux] for EPI_DTANH_BF16
  int ld_aux;
  float* colsum;           // EPI_DTANH_BF16: [N] += column sums of the bf16 output (bias gradient of the layer below), or null
};

template <int BN>
struct Smem {
  static constexpr int A_BYTES = BM * BK * 2;   // 16 KB
  static constexpr int B_BYTES = BN * BK * 2;   // 8 / 16 KB
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // ring depth: BN <= 128 -> 3 x 32 KB and two CTAs per SM; BN = 256 -> one CTA per SM, so the same
  // 192 KB in flight take 4 x 48 KB (with 3 the TMA latency was exposed: measured 15 % slower)
  static constexpr int NSTAGES = BN == 256 ? 4 : STAGES;
  static constexpr int TOTAL = NSTAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/ + 2048 /*bias*/ +
                               EPI_WARPS * 32 * 80 /*epilogue staging*/;
};


constexpr bool FWD_DIRECT_STORES = true;   // forward epilogue: re-staging through shared memory like dgrad was measured slower (K=64: 37.8 vs 32.0 us)
constexpr int STAGE_PITCH = 80;                       // bytes per staged row: 64 B of bf16 + 16 B pad (conflict-free STS.128)
constexpr int STAGE_BYTES_PER_WARP = 32 * STAGE_PITCH;

// One 32-column chunk of a warp's 32 accumulator rows through the fused epilogue (v = this lane's
// row, 32 fp32 from TMEM). bf16 results are re-staged through shared memory so that every global
// store instruction writes whole 64-byte row segments of 8 rows (4x fewer L1TEX wavefronts than
// one 16-byte piece of 32 different rows per instruction, which bound the first version).
// The aux rows of one 32x32 chunk in the coalesced pattern (lane -> row 8k + lane/4, 16-byte piece lane%4).
struct AuxChunk { uint4 y[4]; };
__device__ __forceinline__ AuxChunk load_aux_chunk(const GemmArgs& g, int m_base, int lane, int col) {
  AuxChunk a;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = k * 8 + (lane >> 2), c16 = lane & 3;
    a.y[k] = make_uint4(0, 0, 0, 0);
    if (m_base + r < g.M) a.y[k] = __ldg(reinterpret_cast<const uint4*>(g.aux + (size_t)(m_base + r) * g.ld_aux + col) + c16);
  }
  return a;
}

template <int EPI>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[32], int m_base, int lane, int col, const GemmArgs& g,
                                               const float* bias_s, bool bias_in_smem, uint8_t* stage,
                                               const AuxChunk* pre = nullptr, float* colsum_s = nullptr) {
  const int row = m_base + lane;
  if (EPI == EPI_BIAS_TANH_BF16 || EPI == EPI_DTANH_BF16) {
    uint32_t packed[16];
    if (EPI == EPI_BIAS_TANH_BF16) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 bv = bias_in_smem ? *reinterpret_cast<const float4*>(bias_s + col + 4 * j)
                                       : __ldg(reinterpret_cast<const float4*>(g.bias + col + 4 * j));
        const float a = tanh_fast(__uint_as_float(v[4 * j]) + bv.x);
        const float b = tanh_fast(__uint_as_float(v[4 * j + 1]) + bv.y);
        const float c2 = tanh_fast(__uint_as_float(v[4 * j + 2]) + bv.z);
        const float d = tanh_fast(__uint_as_float(v[4 * j + 3]) + bv.w);
        __nv_bfloat162 p = __floats2bfloat162_rn(a, b), q2 = __floats2bfloat162_rn(c2, d);
        packed[2 * j] = *reinterpret_cast<uint32_t*>(&p);
        packed[2 * j + 1] = *reinterpret_cast<uint32_t*>(&q2);
      }
    } else {
      // aux tile (the activations whose tanh' multiplies the accumulator): coalesced 64-byte row
      // segments -> shared memory -> each lane reads back its own row
      __syncwarp();
      const AuxChunk aux = pre ? *pre : load_aux_chunk(g, m_base, lane, col);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = k * 8 + (lane >> 2), c16 = lane & 3;
        *reinterpret_cast<uint4*>(stage + r * STAGE_PITCH + c16 * 16) = aux.y[k];
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint4 y4 = *reinterpret_cast<const uint4*>(stage + lane * STAGE_PITCH + j * 16);
        const uint32_t yy[4] = {y4.x, y4.y, y4.z, y4.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const __nv_bfloat162 y2 = *reinterpret_cast<const __nv_bfloat162*>(&yy[i]);
          const float ya = __bfloat162float(y2.x), yb = __bfloat162float(y2.y);
          const float a = __uint_as_float(v[8 * j + 2 * i]) * (1.0f - ya * ya);
          const float b = __uint_as_float(v[8 * j + 2 * i + 1]) * (1.0f - yb * yb);
          __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
          packed[4 * j + i] = *reinterpret_cast<uint32_t*>(&p);
        }
      }
      __syncwarp();
    }
    if (EPI == EPI_BIAS_TANH_BF16 && FWD_DIRECT_STORES) {  // each lane writes 16-byte pieces of its own row
      if (row < g.M) {
        uint4* o4 = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(g.out) + (size_t)row * g.ldo + col);
#pragma unroll
        for (int j = 0; j < 4; ++j) o4[j] = make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
      }
      return;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j)
      *reinterpret_cast<uint4*>(stage + lane * STAGE_PITCH + j * 16) =
          make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
    __syncwarp();
    __nv_bfloat16* obase = reinterpret_cast<__nv_bfloat16*>(g.out) + col;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int r = k * 8 + (lane >> 2), c16 = lane & 3;
      const uint4 o = *reinterpret_cast<const uint4*>(stage + r * STAGE_PITCH + c16 * 16);
      if (m_base + r < g.M) *(reinterpret_cast<uint4*>(obase + (size_t)(m_base + r) * g.ldo) + c16) = o;
    }
    if (colsum_s) {  // bias gradient of the layer below: column sums of the (bf16-rounded) tile, lane = column
      float sum = 0.0f;  // (rows past M were computed from zero-filled operands and hold zeros)
#pragma unroll
      for (int r = 0; r < 32; ++r)
        sum += __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(stage + r * STAGE_PITCH + 2 * lane));
      atomicAdd(colsum_s + col + lane, sum);
    }
    __syncwarp();
  } else if (EPI == EPI_ATOMIC_F32) {
    if (row < g.M) {
      float* orow = reinterpret_cast<float*>(g.out) + (size_t)row * g.ldo + col;
#pragma unroll
      for (int i = 0; i < 32; i += 4)
        red_add_v4(orow + i, __uint_as_float(v[i]), __uint_as_float(v[i + 1]), __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
    }
  } else {
    if (row < g.M) {
      float* orow = reinterpret_cast<float*>(g.out) + (size_t)row * g.ldo + col;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float4 o;
        o.x = __uint_as_float(v[4 * j]) + (g.bias ? __ldg(g.bias + col + 4 * j) : 0.0f);
        o.y = __uint_as_float(v[4 * j + 1]) + (g.bias ? __ldg(g.bias + col + 4 * j + 1) : 0.0f);
        o.z = __uint_as_float(v[4 * j + 2]) + (g.bias ? __ldg(g.bias + col + 4 * j + 2) : 0.0f);
        o.w = __uint_as_float(v[4 * j + 3]) + (g.bias ? __ldg(g.bias + col + 4 * j + 3) : 0.0f);
        reinterpret_cast<float4*>(orow)[j] = o;
      }
    }
  }
}

// Persistent kernel: each CTA walks tiles t = blockIdx.x, blockIdx.x + gridDim.x, ... (n-tile fastest, so
// CTAs working at the same time share A rows through L2). The accumulator is double-buffered in TMEM
// (2 x BN columns): the MMA warp fills buffer (i+1)&1 while the epilogue warps drain buffer i&1, and the
// TMA producer runs ahead across tile boundaries through the smem ring.
template <int BN, int EPI, bool MN>
__global__ void __launch_bounds__(THREADS, 2)
k_gemm_tn(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
          const __grid_constant__ GemmArgs g) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Smem<BN>::NSTAGES * Smem<BN>::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + Smem<BN>::NSTAGES;
  uint64_t* tfull_bar = empty_bar + Smem<BN>::NSTAGES;   // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;       // [2] accumulator drained
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
  float* bias_s = reinterpret_cast<float*>(smem + Smem<BN>::NSTAGES * Smem<BN>::STAGE_BYTES + 256);  // [<= 512]
  uint8_t* stage = smem + Smem<BN>::NSTAGES * Smem<BN>::STAGE_BYTES + 256 + 2048 + (((threadIdx.x >> 5) + EPI_WARPS - 2) % EPI_WARPS) * STAGE_BYTES_PER_WARP;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = g.N / BN, m_tiles = (g.M + BM - 1) / BM;
  const int tiles_per_split = n_tiles * m_tiles;
  const int total_tiles = tiles_per_split * g.splits;
  const int total_kb = g.K / BK;
  const int t_begin = blockIdx.x, t_step = gridDim.x;

  if (threadIdx.x == 0) {
    for (int s = 0; s < Smem<BN>::NSTAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull_bar[b], 1); mbar_init(&tempty_bar[b], EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * BN);
  const bool bias_in_smem = (EPI == EPI_BIAS_TANH_BF16 || EPI == EPI_BIAS_F32) && g.bias != nullptr && g.N <= 512;
  if (bias_in_smem)  // the whole bias vector once per CTA: the epilogue reads it as broadcast float4s
    for (int i = threadIdx.x; i < g.N; i += THREADS) bias_s[i] = __ldg(g.bias + i);
  // dgrad: per-CTA column sums of the produced tiles live in the (otherwise unused) bias buffer
  float* colsum_s = (EPI == EPI_DTANH_BF16 && g.colsum != nullptr) ? bias_s : nullptr;
  if (colsum_s)
    for (int i = threadIdx.x; i < g.N; i += THREADS) colsum_s[i] = 0.0f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer
      uint32_t s = 0, ph = 0;  // ring position and phase (continue across tiles; no divisions on this path)
      for (int t = t_begin; t < total_tiles; t += t_step) {
        const int split = t / tiles_per_split, r = t % tiles_per_split;
        const int m0 = (r / n_tiles) * BM, n0 = (r % n_tiles) * BN;
        const int kb0 = split * g.k_blocks_per_split;
        const int nkb = min(g.k_blocks_per_split, total_kb - kb0);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* sa = smem + s * Smem<BN>::STAGE_BYTES;
          uint8_t* sb = sa + Smem<BN>::A_BYTES;
          mbar_expect_tx(&full_bar[s], Smem<BN>::STAGE_BYTES);
          if (!MN) {
            tma_load_2d(sa, &map_a, &full_bar[s], (kb0 + kb) * BK, m0);
            tma_load_2d(sb, &map_b, &full_bar[s], (kb0 + kb) * BK, n0);
          } else {  // source tensors are [K, M] / [K, N]: 64 x 64 boxes, inner coordinate = m / n
#pragma unroll
            for (int i = 0; i < BM / 64; ++i) tma_load_2d(sa + i * 8192, &map_a, &full_bar[s], m0 + 64 * i, (kb0 + kb) * BK);
#pragma unroll
            for (int i = 0; i < BN / 64; ++i) tma_load_2d(sb + i * 8192, &map_b, &full_bar[s], n0 + 64 * i, (kb0 + kb) * BK);
          }
          if (++s == Smem<BN>::NSTAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {  // ---- MMA issuer
      constexpr uint32_t idesc = make_idesc(BM, BN, MN);
      uint32_t s = 0, ph = 0, lt = 0;
      for (int t = t_begin; t < total_tiles; t += t_step, ++lt) {
        const int split = t / tiles_per_split;
        const int kb0 = split * g.k_blocks_per_split;
        const int nkb = min(g.k_blocks_per_split, total_kb - kb0);
        const uint32_t buf = lt & 1, bph = (lt >> 1) & 1;
        mbar_wait(&tempty_bar[buf], bph ^ 1);  // the epilogue has drained this accumulator buffer
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * Smem<BN>::STAGE_BYTES);
          const uint64_t adesc = MN ? make_desc_mn128(sa) : make_desc_k128(sa);
          const uint64_t bdesc = MN ? make_desc_mn128(sa + Smem<BN>::A_BYTES) : make_desc_k128(sa + Smem<BN>::A_BYTES);
          // per K=16 step: K-major +32 B inside the swizzle row (>>4 = 2); MN-major +16 rows = 2048 B (>>4 = 128)
          constexpr uint64_t kstep = MN ? 128 : 2;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_bf16(tmem_d, adesc + kstep * k, bdesc + kstep * k, idesc, (kb | k) != 0);
          umma_commit(&empty_bar[s]);  // frees the smem stage when these MMAs retire
          if (++s == Smem<BN>::NSTAGES) { s = 0; ph ^= 1; }
        }
        umma_commit(&tfull_bar[buf]);  // accumulator complete
      }
    }
  } else {
    // ---- epilogue: warp w may touch TMEM lanes [32*(w%4), +32)
    const int q = warp & 3;                              // TMEM lane quarter this warp may touch
    constexpr int COLS_PER_WARP = BN / (EPI_WARPS / 4);  // column share of this warp within the quarter
    const int c_begin = ((warp - 2) >> 2) * COLS_PER_WARP;
    uint32_t lt = 0;
    AuxChunk aux_next[4];
    for (int t = t_begin; t < total_tiles; t += t_step, ++lt) {
      const int r = t % tiles_per_split;
      const int m0 = (r / n_tiles) * BM, n0 = (r % n_tiles) * BN;
      const uint32_t buf = lt & 1, bph = (lt >> 1) & 1;
      if (EPI == EPI_DTANH_BF16 && BN == 128 && EPI_WARPS == 4) {
        // The aux rows come from DRAM: issued when they are needed, every chunk exposed a full memory
        // round trip (ncu: long_scoreboard 8 per issue, tensor pipe 19 % at K = 256). They are kept one
        // tile ahead in registers instead — chunk c of the NEXT tile is requested as soon as chunk c of
        // this tile has been copied to the staging buffer.
        if (lt == 0) {
#pragma unroll
          for (int ci = 0; ci < 4; ++ci) aux_next[ci] = load_aux_chunk(g, m0 + q * 32, lane, n0 + 32 * ci);
        }
        const int tn = t + t_step;
        const int rn = tn % tiles_per_split;
        const int m0n = (rn / n_tiles) * BM, n0n = (rn % n_tiles) * BN;
        mbar_wait(&tfull_bar[buf], bph);
        tc_fence_after();
#pragma unroll
        for (int ci = 0; ci < 4; ++ci) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + (uint32_t)(32 * ci), v);
          const AuxChunk cur = aux_next[ci];
          if (tn < total_tiles) aux_next[ci] = load_aux_chunk(g, m0n + q * 32, lane, n0n + 32 * ci);
          epilogue_chunk<EPI>(v, m0 + q * 32, lane, n0 + 32 * ci, g, bias_s, bias_in_smem, stage, &cur, colsum_s);
        }
      } else {
        mbar_wait(&tfull_bar[buf], bph);
        tc_fence_after();
#pragma unroll 1
        for (int c = c_begin; c < c_begin + COLS_PER_WARP; c += 32) {
          uint32_t v[32];
          tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + (uint32_t)c, v);
          epilogue_chunk<EPI>(v, m0 + q * 32, lane, n0 + c, g, bias_s, bias_in_smem, stage, nullptr, colsum_s);
        }
      }
      // all TMEM reads of this warp are complete (tcgen05.wait::ld): hand the buffer back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (colsum_s)
    for (int i = threadIdx.x; i < g.N; i += THREADS) atomicAdd(g.colsum + i, colsum_s[i]);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * BN);
  }
}

// ---------------------------------------------------------------------------------------------
// CTA-pair kernel for the forward GEMMs (K-major, N % 256 == 0): tcgen05 `cta_group::2`.
// Two CTAs on the two SMs of a TPC (a cluster of 2) compute one 256 x 256 output tile: each CTA
// stages ITS 128 rows of A and ITS 128 of the 256 B rows (N) per k-block — 32 KB per stage for 4.2 MFLOP
// of its tensor core, 131 FLOP per staged byte like the weight-stationary kernel, but without the
// 128 KB resident weight slice, so the ring is 6 x 32 KB deep instead of 4 x 16 KB: the streaming of
// the activation tiles was latency-bound by the bytes in flight (K = 512: 767 TFLOP/s with 64 KB in
// flight per SM). One thread of the leader CTA (cluster rank 0) issues the MMAs for both tensor
// cores (M = 256: rows 0-127 accumulate in the leader's TMEM, rows 128-255 in the peer's, same
// columns); both CTAs' TMA loads complete on the LEADER's full barrier (the leader arms it for
// both halves); tcgen05.commit multicasts the "stage free" and "accumulator ready" arrivals to both
// CTAs; the peer's epilogue warps hand the accumulator buffer back by arriving on the leader's
// barrier across the cluster. Epilogue as in k_gemm_ws: bias + tanh -> bf16 -> swizzled staging box
// -> bulk tensor store, TMEM loads software-pipelined; accumulators double-buffered (2 x 256 columns).
// ---------------------------------------------------------------------------------------------
constexpr int P2_BN = 256;
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address: the leader's copy
// Shared memory of the pair kernel. EW = epilogue warps: 4 (one per TMEM lane quarter, all 256 columns) where the
// mainloop binds (K = 512), 8 (two per quarter, 128 columns each) where the epilogue binds (K <= 256: few MMAs per
// tile, the same bias + tanh / tanh' + store work). Each epilogue warp owns 32 x 64 staging boxes (128-byte rows,
// 128B-swizzled tensor-map boxes): two for the output (one being stored, one being filled; one with 8 warps in dgrad)
// and, in dgrad, two for the tanh' operand (the activations of the layer below, fetched by TMA one box ahead).
template <int EPI, int EW>
struct SmemPair {
  static constexpr int A_BYTES = BM * BK * 2, B_BYTES = 128 * BK * 2, STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = EPI == EPI_DTANH_BF16 ? (EW == 8 ? 3 : 4) : (EW == 8 ? 4 : 5);
  static constexpr int BOX = 32 * 128;
  static constexpr int OUT_BOXES = (EPI == EPI_DTANH_BF16 && EW == 8) ? 1 : 2;
  static constexpr int OUT_STAGE = OUT_BOXES * BOX;
  static constexpr int AUX_STAGE = EPI == EPI_DTANH_BF16 ? 2 * BOX : 0;
  static constexpr int TOTAL = STAGES * STAGE_BYTES + EW * (OUT_STAGE + AUX_STAGE) + 256 + 2048 + 1024;
  static_assert(TOTAL <= 232448, "dynamic shared memory per CTA");
};
__device__ __forceinline__ void tma_store_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint64_t* leader_bar, int c_inner, int c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(leader_bar) & PEER_BIT_MASK), "r"(c_inner), "r"(c_outer) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {  // arrives on `bar` of BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {  // arrive on the leader CTA's copy of `bar`
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}

template <int EPI, int EW>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
k_gemm_pair(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
            const __grid_constant__ CUtensorMap map_o, const __grid_constant__ CUtensorMap map_x,
            const __grid_constant__ GemmArgs g) {
  static_assert(EPI == EPI_BIAS_TANH_BF16 || EPI == EPI_DTANH_BF16, "forward or dgrad epilogue");
  static_assert(EW == 4 || EW == 8, "one or two epilogue warps per TMEM lane quarter");
  using SM = SmemPair<EPI, EW>;
  constexpr int P2_STAGES = SM::STAGES, NTHREADS = 64 + 32 * EW;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* out_stage = smem + P2_STAGES * SM::STAGE_BYTES;  // 1024-byte aligned (and so is every box after it)
  uint8_t* aux_stage = out_stage + EW * SM::OUT_STAGE;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(aux_stage + EW * SM::AUX_STAGE);
  uint64_t* empty_bar = full_bar + P2_STAGES;
  uint64_t* tfull_bar = empty_bar + P2_STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint64_t* aux_bar = tempty_bar + 2;   // [EW][2] tanh'-operand box landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(aux_bar + 2 * EW);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);   // forward: bias; dgrad: column sums
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const bool leader = rank == 0;
  const int n_tiles = g.N / P2_BN, m_tiles = (g.M + 2 * BM - 1) / (2 * BM);
  const int total_tiles = n_tiles * m_tiles, nkb = g.K / BK;
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < P2_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull_bar[b], 1); mbar_init(&tempty_bar[b], 2 * EW); }
    for (int b = 0; b < 2 * EW; ++b) mbar_init(&aux_bar[b], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // the same warp of both CTAs allocates all 512 columns of the pair's tensor memory
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  for (int i = threadIdx.x; i < g.N; i += NTHREADS)   // N <= 512 (checked by the host)
    bias_s[i] = EPI == EPI_BIAS_TANH_BF16 ? __ldg(g.bias + i) : 0.0f;
  tc_fence_before();
  __syncthreads();
  cluster_sync();  // the peer's barriers are initialised before anything is signalled to them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {  // ---- TMA producer (both CTAs): own 128 rows of A, own 128 rows of B
      uint32_t s = 0, ph = 0;
      for (int t = pair; t < total_tiles; t += npairs) {
        const int m0 = (t / n_tiles) * (2 * BM) + rank * BM, n0 = (t % n_tiles) * P2_BN + rank * 128;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1);
          uint8_t* sa = smem + s * SM::STAGE_BYTES;
          if (leader) mbar_expect_tx(&full_bar[s], 2 * SM::STAGE_BYTES);  // both CTAs' halves land on this barrier
          tma_load_2d_pair(sa, &map_a, &full_bar[s], kb * BK, m0);
          tma_load_2d_pair(sa + SM::A_BYTES, &map_b, &full_bar[s], kb * BK, n0);
          if (++s == P2_STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && leader) {  // ---- MMA issuer: one thread for both tensor cores
      constexpr uint32_t idesc = make_idesc(2 * BM, P2_BN, false);
      uint32_t s = 0, ph = 0, lt = 0;
      for (int t = pair; t < total_tiles; t += npairs, ++lt) {
        const uint32_t buf = lt & 1, bph = (lt >> 1) & 1;
        mbar_wait(&tempty_bar[buf], bph ^ 1);  // both CTAs' epilogues have drained this buffer
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + buf * P2_BN;
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + s * SM::STAGE_BYTES);
          const uint64_t adesc = make_desc_k128(sa), bdesc = make_desc_k128(sa + SM::A_BYTES);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k)
            umma_bf16_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0);
          umma_commit_pair(&empty_bar[s]);  // the stage is free in both CTAs when these MMAs retire
          if (++s == P2_STAGES) { s = 0; ph ^= 1; }
        }
        umma_commit_pair(&tfull_bar[buf]);  // accumulator complete, in both CTAs
      }
    }
  } else {
    // ---- epilogue (both CTAs): this CTA's 128 rows x 256 columns; warp -> TMEM lane quarter q (a warp may only touch
    // the lanes of quarter warp % 4) and, with 8 warps, the lower or upper 128 columns
    const int q = warp & 3, ew = warp - 2;
    constexpr int CHUNKS = (P2_BN / 32) / (EW / 4);     // 32-column chunks per warp and tile
    const int c0 = (EW == 8 ? (ew >> 2) : 0) * CHUNKS;  // first chunk of this warp
    uint8_t* stage = out_stage + ew * SM::OUT_STAGE;
    uint8_t* xstage = aux_stage + ew * SM::AUX_STAGE;
    uint64_t* xbar = aux_bar + 2 * ew;
    uint32_t lt = 0, xbox = 0;   // xbox: boxes of the tanh' operand consumed so far (buffer = xbox & 1, phase = (xbox >> 1) & 1)
    if (EPI == EPI_DTANH_BF16 && lane == 0 && pair < total_tiles) {   // the first box of the first tile
      mbar_expect_tx(&xbar[0], SM::BOX);
      tma_load_2d(xstage, &map_x, &xbar[0], (pair % n_tiles) * P2_BN + 32 * c0, (pair / n_tiles) * (2 * BM) + rank * BM + q * 32);
    }
    for (int t = pair; t < total_tiles; t += npairs, ++lt) {
      const int m0 = (t / n_tiles) * (2 * BM) + rank * BM + q * 32, n0 = (t % n_tiles) * P2_BN;
      const uint32_t buf = lt & 1, bph = (lt >> 1) & 1;
      mbar_wait(&tfull_bar[buf], bph);
      tc_fence_after();
      uint32_t v[2][32];
      const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + buf * P2_BN + 32u * c0;
      tmem_ld32_issue(t0, v[0]);
#pragma unroll
      for (int cj = 0; cj < CHUNKS; ++cj) {
        const int ci = c0 + cj;   // (c0 is even: cj and ci have the same parity)
        tmem_ld_wait();
        if (cj + 1 < CHUNKS) tmem_ld32_issue(t0 + 32u * (cj + 1), v[(cj + 1) & 1]);
        uint8_t* box = stage + ((cj >> 1) % SM::OUT_BOXES) * SM::BOX;   // the output boxes alternate
        if ((cj & 1) == 0) {  // the store that last used this box has read it out of shared memory
          if (lane == 0) { if (SM::OUT_BOXES == 2) tma_store_wait_read1(); else tma_store_wait_read(); }
          __syncwarp();
        }
        const int col = n0 + 32 * ci;
        const uint8_t* xb = xstage + (xbox & 1) * SM::BOX;   // (dgrad) the box of the tanh' operand for these 64 columns
        if (EPI == EPI_DTANH_BF16 && (ci & 1) == 0) {
          // request the NEXT box (same tile, or the first box of this warp's next tile) into the other buffer —
          // its previous contents were consumed one box ago — then wait for this one
          const bool last = cj + 2 >= CHUNKS;
          const int tn = last ? t + npairs : t;
          if (lane == 0 && tn < total_tiles) {
            const int cn = last ? (tn % n_tiles) * P2_BN + 32 * c0 : col + 64;
            const int rn = last ? (tn / n_tiles) * (2 * BM) + rank * BM + q * 32 : m0;
            mbar_expect_tx(&xbar[(xbox + 1) & 1], SM::BOX);
            tma_load_2d(xstage + ((xbox + 1) & 1) * SM::BOX, &map_x, &xbar[(xbox + 1) & 1], cn, rn);
          }
          mbar_wait(&xbar[xbox & 1], (xbox >> 1) & 1);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t* x = &v[cj & 1][8 * j];
          const int k = (cj & 1) * 4 + j;
          float o[8];
          if (EPI == EPI_BIAS_TANH_BF16) {
            const float4 b0 = *reinterpret_cast<const float4*>(bias_s + col + 8 * j);
            const float4 b1 = *reinterpret_cast<const float4*>(bias_s + col + 8 * j + 4);
            const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i) o[i] = tanh_fast(__uint_as_float(x[i]) + bb[i]);
          } else {  // acc * (1 - y^2), y = this row's activations of the layer below (same swizzled box layout)
            const uint4 y4 = *reinterpret_cast<const uint4*>(xb + lane * 128 + ((k ^ (lane & 7)) << 4));
            const uint32_t yy[4] = {y4.x, y4.y, y4.z, y4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const __nv_bfloat162 y2 = *reinterpret_cast<const __nv_bfloat162*>(&yy[i]);
              const float ya = __bfloat162float(y2.x), yb = __bfloat162float(y2.y);
              o[2 * i] = __uint_as_float(x[2 * i]) * (1.0f - ya * ya);
              o[2 * i + 1] = __uint_as_float(x[2 * i + 1]) * (1.0f - yb * yb);
            }
          }
          __nv_bfloat162 p0 = __floats2bfloat162_rn(o[0], o[1]), p1 = __floats2bfloat162_rn(o[2], o[3]);
          __nv_bfloat162 p2 = __floats2bfloat162_rn(o[4], o[5]), p3 = __floats2bfloat162_rn(o[6], o[7]);
          *reinterpret_cast<uint4*>(box + lane * 128 + ((k ^ (lane & 7)) << 4)) =
              make_uint4(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1),
                         *reinterpret_cast<uint32_t*>(&p2), *reinterpret_cast<uint32_t*>(&p3));
        }
        if (ci & 1) {
          if (EPI == EPI_DTANH_BF16) {
            __syncwarp();
            if (g.colsum != nullptr) {
              // bias gradient of the layer below: column sums of the (bf16-rounded) box, two columns per lane
              float s0 = 0.0f, s1 = 0.0f;  // (rows past M were computed from zero-filled operands and hold zeros)
#pragma unroll
              for (int r = 0; r < 32; ++r) {
                const __nv_bfloat162 e = *reinterpret_cast<const __nv_bfloat162*>(box + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + 4 * (lane & 3));
                s0 += __bfloat162float(e.x); s1 += __bfloat162float(e.y);
              }
              atomicAdd(bias_s + n0 + 32 * (ci - 1) + 2 * lane, s0);
              atomicAdd(bias_s + n0 + 32 * (ci - 1) + 2 * lane + 1, s1);
            }
            ++xbox;
          }
          fence_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&map_o, box, n0 + 32 * (ci - 1), m0);
            tma_store_commit();
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&tempty_bar[buf]);  // (the leader's own warps arrive locally through the same address)
    }
    if (lane == 0) tma_store_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (EPI == EPI_DTANH_BF16 && g.colsum != nullptr)
    for (int i = threadIdx.x; i < g.N; i += NTHREADS) atomicAdd(g.colsum + i, bias_s[i]);
  cluster_sync();  // no CTA leaves while its peer can still signal it or read its shared memory
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

template <int EPI, int EW>
static cudaError_t launch_pair(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mo, const CUtensorMap& mx,
                               const GemmArgs& g, cudaStream_t st) {
  static bool configured = false;
  static int sms = 148;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(k_gemm_pair<EPI, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, SmemPair<EPI, EW>::TOTAL);
    if (e != cudaSuccess) return e;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    configured = true;
  }
  const long long tiles = (long long)((g.M + 2 * BM - 1) / (2 * BM)) * (g.N / P2_BN);
  unsigned grid = (unsigned)std::min<long long>(2 * tiles, sms & ~1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(64 + 32 * EW); cfg.dynamicSmemBytes = SmemPair<EPI, EW>::TOTAL; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_gemm_pair<EPI, EW>, ma, mb, mo, mx, g);
}

template <int BN, int EPI, bool MN>
static cudaError_t launch(const CUtensorMap& ma, const CUtensorMap& mb, const GemmArgs& g, int splits, cudaStream_t st) {
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(k_gemm_tn<BN, EPI, MN>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Smem<BN>::TOTAL);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  static int max_ctas = 0;
  if (max_ctas == 0) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    max_ctas = 2 * sms;  // two resident CTAs per SM (smem and TMEM both allow exactly two)
  }
  const int resident = BN == 256 ? max_ctas / 2 : max_ctas;  // 128x256 tiles: 144 KB smem + all 512 TMEM columns
  const long long tiles = (long long)((g.M + BM - 1) / BM) * (g.N / BN) * splits;
  unsigned grid = (unsigned)std::min<long long>(tiles, resident);
  k_gemm_tn<BN, EPI, MN><<<grid, THREADS, Smem<BN>::TOTAL, st>>>(ma, mb, g);
  return cudaGetLastError();
}

}  // namespace tc

namespace tc {

// Column sums of a bf16 [M, N] matrix into fp32 out[N] (+=): the bias gradients db = sum_m dZ[m, :].
// Each warp streams 128-byte row segments (64 columns), 8 warps per block take interleaved rows.
__global__ void __launch_bounds__(256)
k_colsum_bf16(const __nv_bfloat16* __restrict__ x, int ld, int M, int N, float* __restrict__ out, int rows_per_block) {
  __shared__ float red[8][64];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c0 = blockIdx.x * 64 + 2 * lane;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(M, r0 + rows_per_block);
  float a0 = 0.f, a1 = 0.f;
  if (c0 < N) {
#pragma unroll 4
    for (int r = r0 + w; r < r1; r += 8) {
      const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(x + (size_t)r * ld + c0);
      a0 += __bfloat162float(v.x); a1 += __bfloat162float(v.y);
    }
  }
  red[w][2 * lane] = a0; red[w][2 * lane + 1] = a1;
  __syncthreads();
  if (threadIdx.x < 64 && blockIdx.x * 64 + threadIdx.x < N) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += red[k][threadIdx.x];
    atomicAdd(out + blockIdx.x * 64 + threadIdx.x, s);
  }
}

// dst[m, 0:ncol_pad] (bf16) = [ src[idx ? idx[m] : m, 0:ncol] (f32), zeros ]: the minibatch gather
// (ppo…:314 `b_obs[mb_inds]`) fused with the bf16 conversion and the 52 -> 64 column padding.
__global__ void __launch_bounds__(256)
k_gather_pad_bf16(const float* __restrict__ src, const long long* __restrict__ idx, int M, int ncol, int ncol_pad,
                  __nv_bfloat16* __restrict__ dst) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per_row = ncol_pad / 2;
  if (t >= (long long)M * per_row) return;
  const int m = (int)(t / per_row), c = 2 * (int)(t % per_row);
  const long long r = idx ? idx[m] : m;
  const float a = c < ncol ? __ldg(src + r * ncol + c) : 0.f;
  const float b = c + 1 < ncol ? __ldg(src + r * ncol + c + 1) : 0.f;
  *reinterpret_cast<__nv_bfloat162*>(dst + (size_t)m * ncol_pad + c) = __floats2bfloat162_rn(a, b);
}

// ---- the 256 -> {1,2,6} output head (Linear without activation, ppo…:138,151) on CUDA cores -------
// One warp per row, lane l owns columns 8l..8l+7 of the 256-wide hidden vector (one 16-byte load).
template <int NO>
__global__ void __launch_bounds__(256)
k_head_fwd(const __nv_bfloat16* __restrict__ h, int ldh, const float* __restrict__ W, const float* __restrict__ b,
           float* __restrict__ out, int M) {
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  float w[NO][8];
#pragma unroll
  for (int j = 0; j < NO; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) w[j][c] = __ldg(W + j * 256 + 8 * lane + c);
  constexpr int U = 4;  // rows in flight per warp (each row is one 16-byte load per lane)
  for (int m0 = warp; m0 < M; m0 += U * nwarps) {
    uint4 raws[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = m0 + u * nwarps;
      if (m < M) raws[u] = *reinterpret_cast<const uint4*>(h + (size_t)m * ldh + 8 * lane);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = m0 + u * nwarps;
      if (m >= M) break;
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raws[u]);
      float x[8];
#pragma unroll
      for (int c = 0; c < 4; ++c) { x[2 * c] = __bfloat162float(h2[c].x); x[2 * c + 1] = __bfloat162float(h2[c].y); }
#pragma unroll
      for (int j = 0; j < NO; ++j) {
        float acc = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) acc = fmaf(x[c], w[j][c], acc);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (lane == 0) out[(size_t)m * NO + j] = acc + __ldg(b + j);
      }
    }
  }
}

// Backward of the head fused with the tanh' of the last hidden layer:
//   dZ[m,c] = (sum_j dout[m,j] W[j,c]) * (1 - h[m,c]^2)   (bf16 out)
//   dW[j,c] += sum_m dout[m,j] h[m,c];   db[j] += sum_m dout[m,j]
template <int NO>
__global__ void __launch_bounds__(256, NO <= 2 ? 3 : 1)
k_head_bwd(const float* __restrict__ dout, const __nv_bfloat16* __restrict__ h, int ldh, const float* __restrict__ W,
           __nv_bfloat16* __restrict__ dz, int ldz, float* __restrict__ dW, float* __restrict__ db,
           float* __restrict__ dz_colsum, int M) {
  __shared__ float red[8][NO][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  float w[NO][8], gw[NO][8], gb[NO], gz[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) gz[c] = 0.f;
#pragma unroll
  for (int j = 0; j < NO; ++j) {
    gb[j] = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) { w[j][c] = __ldg(W + j * 256 + 8 * lane + c); gw[j][c] = 0.f; }
  }
  // U rows per warp in flight: with one row per iteration every row was a DRAM round trip on the warp's
  // critical path (55 rows x ~1.5 us = 98 us for 134 MB of traffic). Rows are consumed in the same
  // ascending order as before, so the accumulated sums are unchanged.
  constexpr int U = NO >= 6 ? 2 : 4;  // (NO = 6 at U = 4 needs 192 registers: one CTA per SM)
  for (int m0 = warp; m0 < M; m0 += U * nwarps) {
    uint4 raws[U];
    float ds[U][NO];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = m0 + u * nwarps;
      if (m < M) {
        raws[u] = *reinterpret_cast<const uint4*>(h + (size_t)m * ldh + 8 * lane);
#pragma unroll
        for (int j = 0; j < NO; ++j) ds[u][j] = __ldg(dout + (size_t)m * NO + j);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int m = m0 + u * nwarps;
      if (m >= M) break;
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&raws[u]);
      float x[8], g[8], d[NO];
#pragma unroll
      for (int c = 0; c < 4; ++c) { x[2 * c] = __bfloat162float(h2[c].x); x[2 * c + 1] = __bfloat162float(h2[c].y); }
#pragma unroll
      for (int j = 0; j < NO; ++j) { d[j] = ds[u][j]; gb[j] += d[j]; }
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float acc = 0.f;
#pragma unroll
        for (int j = 0; j < NO; ++j) { acc = fmaf(d[j], w[j][c], acc); gw[j][c] = fmaf(d[j], x[c], gw[j][c]); }
        g[c] = acc * (1.0f - x[c] * x[c]);
      }
      uint4 o;
      __nv_bfloat162 p0 = __floats2bfloat162_rn(g[0], g[1]), p1 = __floats2bfloat162_rn(g[2], g[3]);
      __nv_bfloat162 p2 = __floats2bfloat162_rn(g[4], g[5]), p3 = __floats2bfloat162_rn(g[6], g[7]);
      o.x = *reinterpret_cast<uint32_t*>(&p0); o.y = *reinterpret_cast<uint32_t*>(&p1);
      o.z = *reinterpret_cast<uint32_t*>(&p2); o.w = *reinterpret_cast<uint32_t*>(&p3);
      *reinterpret_cast<uint4*>(dz + (size_t)m * ldz + 8 * lane) = o;
      // bias gradient of the last hidden layer = column sums of dz as stored (bf16-rounded)
      gz[0] += __bfloat162float(p0.x); gz[1] += __bfloat162float(p0.y); gz[2] += __bfloat162float(p1.x);
      gz[3] += __bfloat162float(p1.y); gz[4] += __bfloat162float(p2.x); gz[5] += __bfloat162float(p2.y);
      gz[6] += __bfloat162float(p3.x); gz[7] += __bfloat162float(p3.y);
    }
  }
#pragma unroll
  for (int j = 0; j < NO; ++j)
#pragma unroll
    for (int c = 0; c < 8; ++c) red[wib][j][8 * lane + c] = gw[j][c];
  __syncthreads();
  for (int i = threadIdx.x; i < NO * 256; i += blockDim.x) {
    const int j = i / 256, c = i % 256;
    float sacc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc += red[k][j][c];
    atomicAdd(dW + j * 256 + c, sacc);
  }
  if (lane == 0)
#pragma unroll
    for (int j = 0; j < NO; ++j) atomicAdd(db + j, gb[j]);
  if (dz_colsum) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < 8; ++c) red[wib][0][8 * lane + c] = gz[c];
    __syncthreads();
    float sacc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc += red[k][0][threadIdx.x];
    atomicAdd(dz_colsum + threadIdx.x, sacc);
  }
}

}  // namespace tc

extern thread_local std::string g_tc_error;
thread_local std::string g_tc_error;

extern "C" {

VSS_API const char* vss_gemm_last_error(void) { return g_tc_error.c_str(); }

// C[M,N] = epi(op(A) * op(B)^T), bf16 operands, fp32 accumulation on the tensor cores.
//   mn_major = 0: A is [M,K], B is [N,K] row-major (K contiguous) — forward and dgrad.
//   mn_major = 1: A is [K,M], B is [K,N] row-major (the reduction index is the row) — wgrad
//                 dW[N_out,K_in] = sum_batch dZ[batch,N_out] * X[batch,K_in], no transposes needed.
// lda/ldb/ldo/ld_aux in elements (layout rules: include/vss_b200.h). K: multiple of 64, or ragged with mn_major (TMA zero-fills
// rows past K). N multiple of 64. epilogue: see tc::Epilogue. splits > 1 only with EPI_ATOMIC_F32
// (the caller zeroes `out`). Returns 0 or a negative VSS_E_* code (message: vss_gemm_last_error).
VSS_API int vss_gemm_bf16_tn(const void* A, int lda, const void* B, int ldb, void* out, int ldo, int M, int N, int K,
                             int epilogue, const float* bias, const void* aux, int ld_aux, int splits, int mn_major,
                             void* stream) {
  return vss_gemm_bf16_tn_colsum(A, lda, B, ldb, out, ldo, M, N, K, epilogue, bias, aux, ld_aux, splits, mn_major,
                                 nullptr, stream);
}

// The same, plus (dgrad epilogue only) colsum[N] += column sums of the bf16 output: the bias gradient of
// the layer below comes out of the GEMM that produces dZ instead of a second pass over it.
VSS_API int vss_gemm_bf16_tn_colsum(const void* A, int lda, const void* B, int ldb, void* out, int ldo, int M, int N,
                                    int K, int epilogue, const float* bias, const void* aux, int ld_aux, int splits,
                                    int mn_major, float* colsum, void* stream) {
  using namespace tc;
  if (colsum && (epilogue != EPI_DTANH_BF16 || mn_major || N > 512)) {
    g_tc_error = "vss_gemm_bf16_tn_colsum: column sums need the dgrad epilogue, K-major operands and N <= 512";
    return VSS_E_INVALID;
  }
  if (!A || !B || !out || M <= 0 || N <= 0 || K <= 0) { g_tc_error = "vss_gemm_bf16_tn: bad argument"; return VSS_E_INVALID; }
  if (epilogue < EPI_BIAS_TANH_BF16 || epilogue > EPI_BIAS_F32 || (mn_major && epilogue != EPI_ATOMIC_F32)) {
    g_tc_error = "vss_gemm_bf16_tn: unsupported epilogue / layout combination"; return VSS_E_INVALID;
  }
  if ((!mn_major && K % BK != 0) || N % 64 != 0 || lda % 8 != 0 || ldb % 8 != 0 || (mn_major && M % 128 != 0)) {
    g_tc_error = "vss_gemm_bf16_tn: K must be a multiple of 64 (K-major), N of 64, lda/ldb of 8, M of 128 (MN-major)";
    return VSS_E_INVALID;
  }
  if (lda < (mn_major ? M : K) || ldb < (mn_major ? N : K)) {
    g_tc_error = "vss_gemm_bf16_tn: lda/ldb smaller than the rows of A/B"; return VSS_E_INVALID;
  }
  // The epilogues store bf16 rows as 16-byte pieces and f32 rows (EPI_BIAS_F32) as float4, read the bias as float4
  // and the tanh' operand as 16-byte pieces: every row start they touch must be 16-byte aligned. The atomic epilogue
  // falls back to scalar reductions on unaligned addresses (red_add_v4).
  const bool bf16_out = epilogue == EPI_BIAS_TANH_BF16 || epilogue == EPI_DTANH_BF16;
  if (ldo < N || (bf16_out && ldo % 8 != 0) || (epilogue == EPI_BIAS_F32 && ldo % 4 != 0) ||
      (epilogue != EPI_ATOMIC_F32 && reinterpret_cast<uintptr_t>(out) % 16 != 0)) {
    g_tc_error = "vss_gemm_bf16_tn: ldo must be >= N (a multiple of 8 for bf16 outputs, of 4 for EPI_BIAS_F32) and out "
                 "16-byte aligned";
    return VSS_E_INVALID;
  }
  if (bias && reinterpret_cast<uintptr_t>(bias) % 16 != 0) {
    g_tc_error = "vss_gemm_bf16_tn: bias must be 16-byte aligned"; return VSS_E_INVALID;
  }
  if (splits < 1) splits = 1;
  if (splits > 1 && epilogue != EPI_ATOMIC_F32) { g_tc_error = "vss_gemm_bf16_tn: split-K needs the atomic epilogue"; return VSS_E_INVALID; }
  if ((epilogue == EPI_BIAS_TANH_BF16 && !bias) || (epilogue == EPI_DTANH_BF16 && !aux)) {
    g_tc_error = "vss_gemm_bf16_tn: missing bias/aux"; return VSS_E_INVALID;
  }
  if (epilogue == EPI_DTANH_BF16 && (ld_aux < N || ld_aux % 8 != 0 || reinterpret_cast<uintptr_t>(aux) % 16 != 0)) {
    g_tc_error = "vss_gemm_bf16_tn: ld_aux must be >= N and a multiple of 8, aux 16-byte aligned"; return VSS_E_INVALID;
  }
  // tile width of the one-CTA kernel: 128 x 256 for the split-K wgrad shapes that do not reach the CTA-pair kernel
  // (short reductions), else 128 x 128 / 128 x 64
  int bn = (N % 128 == 0) ? 128 : 64;
  if (N % 256 == 0 && epilogue == EPI_ATOMIC_F32 && mn_major) bn = 256;
  CUtensorMap ma, mb;
  const bool ok = mn_major ? (make_map(&ma, A, K, M, lda, BK) && make_map(&mb, B, K, N, ldb, BK))
                           : (make_map(&ma, A, M, K, lda, BM) && make_map(&mb, B, N, K, ldb, bn));
  if (!ok) {
    g_tc_error = "vss_gemm_bf16_tn: cuTensorMapEncodeTiled failed"; return VSS_E_CUDA;
  }
  GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.K = (K + BK - 1) / BK * BK;  // ragged K (MN-major only): the TMA zero-fills the tail rows
  const int total_kb = g.K / BK;
  g.k_blocks_per_split = (total_kb + splits - 1) / splits;
  splits = (total_kb + g.k_blocks_per_split - 1) / g.k_blocks_per_split;
  g.splits = splits;
  g.out = out; g.ldo = ldo; g.bias = bias; g.aux = reinterpret_cast<const __nv_bfloat16*>(aux); g.ld_aux = ld_aux;
  g.colsum = colsum;
  cudaStream_t st = (cudaStream_t)stream;
  cudaError_t e = cudaSuccess;
  // forward and dgrad with N a multiple of 256 and enough row tiles: the CTA-pair kernel (tcgen05 cta_group::2)
  if ((epilogue == EPI_BIAS_TANH_BF16 || epilogue == EPI_DTANH_BF16) && !mn_major && splits == 1 && N % 256 == 0 &&
      N <= 512 && M >= 256 * 74) {
    // A: 128-row boxes; B: 128-row boxes (this CTA's half of the 256 columns); out / tanh' operand: 32 x 64 boxes
    CUtensorMap ma2, mb2, mo2, mx2;
    bool ok2 = make_map(&ma2, A, M, K, lda, BM) && make_map(&mb2, B, N, K, ldb, 128) && make_map(&mo2, out, M, N, ldo, 32);
    if (ok2) { if (epilogue == EPI_DTANH_BF16) ok2 = make_map(&mx2, aux, M, N, ld_aux, 32); else mx2 = mo2; }
    if (!ok2) { g_tc_error = "vss_gemm_bf16_tn: cuTensorMapEncodeTiled failed"; return VSS_E_CUDA; }
    // K <= 256: few MMAs per tile, the epilogue binds -> two epilogue warps per TMEM lane quarter (measured at K = 512:
    // 67.2 / 42.3 us with eight warps and a 4-stage ring vs 66.8 / 40.0 us with four warps and 5 stages)
    if (epilogue == EPI_BIAS_TANH_BF16)
      e = K <= 256 ? launch_pair<EPI_BIAS_TANH_BF16, 8>(ma2, mb2, mo2, mx2, g, st) : launch_pair<EPI_BIAS_TANH_BF16, 4>(ma2, mb2, mo2, mx2, g, st);
    else
      e = K <= 256 ? launch_pair<EPI_DTANH_BF16, 8>(ma2, mb2, mo2, mx2, g, st) : launch_pair<EPI_DTANH_BF16, 4>(ma2, mb2, mo2, mx2, g, st);
    if (e != cudaSuccess) { g_tc_error = std::string("vss_gemm_bf16_tn (pair): ") + cudaGetErrorString(e); return VSS_E_CUDA; }
    return VSS_OK;
  }
#define TC_CASE(BNV, EPIV, MNV) \
  if (bn == BNV && epilogue == EPIV && (mn_major != 0) == MNV) e = launch<BNV, EPIV, MNV>(ma, mb, g, splits, st); else
  TC_CASE(128, EPI_BIAS_TANH_BF16, false) TC_CASE(64, EPI_BIAS_TANH_BF16, false)
  TC_CASE(128, EPI_DTANH_BF16, false) TC_CASE(64, EPI_DTANH_BF16, false)
  TC_CASE(128, EPI_ATOMIC_F32, false) TC_CASE(64, EPI_ATOMIC_F32, false)
  TC_CASE(128, EPI_BIAS_F32, false) TC_CASE(64, EPI_BIAS_F32, false)
  TC_CASE(128, EPI_ATOMIC_F32, true) TC_CASE(64, EPI_ATOMIC_F32, true)
  TC_CASE(256, EPI_ATOMIC_F32, true)
  { g_tc_error = "vss_gemm_bf16_tn: unsupported epilogue / layout combination"; return VSS_E_INVALID; }
#undef TC_CASE
  if (e != cudaSuccess) { g_tc_error = std::string("vss_gemm_bf16_tn: ") + cudaGetErrorString(e); return VSS_E_CUDA; }
  return VSS_OK;
}

// out[N] (f32) += column sums of x [M,N] bf16 (row stride ld elements). N even.
VSS_API int vss_colsum_bf16(const void* x, int ld, int M, int N, float* out, void* stream) {
  if (!x || !out || M <= 0 || N <= 0 || (N & 1)) { g_tc_error = "vss_colsum_bf16: bad argument"; return VSS_E_INVALID; }
  if (ld < N || (ld & 1) || reinterpret_cast<uintptr_t>(x) % 4 != 0) {  // rows are read as bf16 pairs
    g_tc_error = "vss_colsum_bf16: ld must be even and >= N, x 4-byte aligned"; return VSS_E_INVALID;
  }
  const int col_blocks = (N + 63) / 64;
  int row_blocks = (148 * 8 + col_blocks - 1) / col_blocks;
  int rows_per_block = (M + row_blocks - 1) / row_blocks;
  rows_per_block = (rows_per_block + 7) / 8 * 8;
  row_blocks = (M + rows_per_block - 1) / rows_per_block;
  tc::k_colsum_bf16<<<dim3(col_blocks, row_blocks), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), ld, M, N, out, rows_per_block);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { g_tc_error = std::string("vss_colsum_bf16: ") + cudaGetErrorString(e); return VSS_E_CUDA; }
  return VSS_OK;
}

// dst [M, ncol_pad] bf16 = pad(src[idx[m] or m, :ncol] f32). idx int64 device array or NULL. ncol_pad even.
VSS_API int vss_gather_pad_bf16(const float* src, const int64_t* idx, int M, int ncol, int ncol_pad, void* dst,
                                void* stream) {
  if (!src || !dst || M <= 0 || ncol <= 0 || ncol_pad < ncol || (ncol_pad & 1)) {
    g_tc_error = "vss_gather_pad_bf16: bad argument"; return VSS_E_INVALID;
  }
  if (reinterpret_cast<uintptr_t>(dst) % 4 != 0) {  // written as bf16 pairs
    g_tc_error = "vss_gather_pad_bf16: dst must be 4-byte aligned"; return VSS_E_INVALID;
  }
  const long long total = (long long)M * (ncol_pad / 2);
  tc::k_gather_pad_bf16<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      src, reinterpret_cast<const long long*>(idx), M, ncol, ncol_pad, reinterpret_cast<__nv_bfloat16*>(dst));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { g_tc_error = std::string("vss_gather_pad_bf16: ") + cudaGetErrorString(e); return VSS_E_CUDA; }
  return VSS_OK;
}

// Output head of the MLP: out [M,n_out] f32 = h [M,256] bf16 * W[n_out,256]^T + b. n_out in {1,2,6}.
VSS_API int vss_head_forward(const void* h, int ldh, const float* W, const float* b, float* out, int M, int n_out,
                             void* stream) {
  if (!h || !W || !b || !out || M <= 0) { g_tc_error = "vss_head_forward: bad argument"; return VSS_E_INVALID; }
  if (ldh < 256 || ldh % 8 != 0 || reinterpret_cast<uintptr_t>(h) % 16 != 0) {  // rows are read as 16-byte pieces
    g_tc_error = "vss_head_forward: ldh must be >= 256 and a multiple of 8, h 16-byte aligned"; return VSS_E_INVALID;
  }
  const __nv_bfloat16* hp = reinterpret_cast<const __nv_bfloat16*>(h);
  const int blocks = std::min((M + 7) / 8, 148 * 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (n_out == 1) tc::k_head_fwd<1><<<blocks, 256, 0, st>>>(hp, ldh, W, b, out, M);
  else if (n_out == 2) tc::k_head_fwd<2><<<blocks, 256, 0, st>>>(hp, ldh, W, b, out, M);
  else if (n_out == 6) tc::k_head_fwd<6><<<blocks, 256, 0, st>>>(hp, ldh, W, b, out, M);
  else { g_tc_error = "vss_head_forward: n_out must be 1, 2 or 6"; return VSS_E_INVALID; }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { g_tc_error = std::string("vss_head_forward: ") + cudaGetErrorString(e); return VSS_E_CUDA; }
  return VSS_OK;
}

// Backward of the head fused with tanh' of the last hidden layer (see k_head_bwd). dW [n_out,256] and
// db [n_out] are accumulated (+=): the caller zeroes them. dz [M,256] bf16.
VSS_API int vss_head_backward(const float* dout, const void* h, int ldh, const float* W, void* dz, int ldz, float* dW,
                              float* db, float* dz_colsum, int M, int n_out, void* stream) {
  if (!dout || !h || !W || !dz || !dW || !db || M <= 0) { g_tc_error = "vss_head_backward: bad argument"; return VSS_E_INVALID; }
  if (ldh < 256 || ldh % 8 != 0 || ldz < 256 || ldz % 8 != 0 || reinterpret_cast<uintptr_t>(h) % 16 != 0 ||
      reinterpret_cast<uintptr_t>(dz) % 16 != 0) {  // h rows are read and dz rows written as 16-byte pieces
    g_tc_error = "vss_head_backward: ldh/ldz must be >= 256 and multiples of 8, h and dz 16-byte aligned";
    return VSS_E_INVALID;
  }
  const __nv_bfloat16* hp = reinterpret_cast<const __nv_bfloat16*>(h);
  __nv_bfloat16* zp = reinterpret_cast<__nv_bfloat16*>(dz);
  // resident blocks per SM: 3 (n_out <= 2, <= 85 registers) or 1 (n_out = 6, 162 registers): one wave, more rows in flight
  const int blocks = std::min((M + 7) / 8, 148 * (n_out <= 2 ? 3 : 1));
  cudaStream_t st = (cudaStream_t)stream;
  if (n_out == 1) tc::k_head_bwd<1><<<blocks, 256, 0, st>>>(dout, hp, ldh, W, zp, ldz, dW, db, dz_colsum, M);
  else if (n_out == 2) tc::k_head_bwd<2><<<blocks, 256, 0, st>>>(dout, hp, ldh, W, zp, ldz, dW, db, dz_colsum, M);
  else if (n_out == 6) tc::k_head_bwd<6><<<blocks, 256, 0, st>>>(dout, hp, ldh, W, zp, ldz, dW, db, dz_colsum, M);
  else { g_tc_error = "vss_head_backward: n_out must be 1, 2 or 6"; return VSS_E_INVALID; }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { g_tc_error = std::string("vss_head_backward: ") + cudaGetErrorString(e); return VSS_E_CUDA; }
  return VSS_OK;
}

}  // extern "C"
