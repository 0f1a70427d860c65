// Decode-step kernels (one new token per sequence, M = batch rows), sm_100a.
//
// The decode step is bandwidth/latency bound (DESIGN.md "decode step"): per layer it streams 11.8 MB of fp32 weights
// (L2-resident across steps) and, per sequence, the self-attention K/V rows written so far plus the 256 hoisted
// cross-attention K/V rows (HBM).  The kernels:
//
//  sgemm_dec_cluster_kernel   exact-fp32 GEMM for M <= 64 rows, the default.  One thread-block CLUSTER (8 CTAs; 16 for
//                      the long-K MLP-out projection) per 64 x 32 output tile splits K; 4 x 4 register tiles, packed FFMA2.
//                      Every CTA pushes the rows owned by rank r into rank r's shared memory (by default one bulk
//                      DSMEM copy per peer onto the peer's mbarrier, operand loads staged under the multiply:
//                      MT3_DEC_PIPE) and each rank sums its rows in rank order (deterministic) and runs the fused epilogue:
//                      RMSNorm factor (statistic computed from the A tiles the GEMM loads anyway, layers.py:613-616),
//                      residual, gated GELU, head-major KV-cache append (fp32 or fp16 cache), per-tile sums of squares
//                      of the output.  (A second warp group per CTA splitting the K chunk once more is written in the
//                      body as G = 2 and measured slower: kDecGroups below.)
//  sgemm_dec_cluster2_kernel  two such GEMMs that read the same inputs in one launch (out-projection + the
//                      cross-attention query projection through a precomposed weight block).
//  sgemm_dec_kernel    the same GEMM without clusters (MT3_DEC_CLUSTER=0 / shapes the cluster kernel does not
//                      tile): K split over gridDim.y CTAs, partial tiles through an L2-resident scratch, the LAST
//                      CTA to arrive for a tile (atomic ticket) sums them in fixed order.
//  dec_attention_bulk_kernel  one query per (sequence, head) over contiguous head-major K/V rows
//                      (kv[b][K|V][head][cap][64], fp32 or fp16 elements).  A producer warp streams 8 KB tiles
//                      (32 fp32 / 64 fp16 keys) with cp.async.bulk (TMA 1-D) into a 6-stage shared-memory ring,
//                      signalled through mbarriers; four consumer warps compute scores (pass 1: K tiles), the
//                      softmax, and P.V (pass 2: V tiles), all in fp32.  Slots >= len are never read -- identical
//                      to the reference's -1e10 mask bias (layers.py:297-322: exp underflows to exactly 0).
#pragma once

#include <cuda_fp16.h>

#include "common.cuh"
#include "gemm_simt.cuh"
#include "tc.cuh"

namespace mt3 {

// ---------------------------------------------------------------------------------------------
// L2 prefetch of head-major K/V rows.  The decode attention kernel reads, per (sequence b, head h), the K rows
// 0..len-1 and then the V rows 0..len-1 of one layer in tiles of KT keys: "virtual tile" j < nt is K tile j, virtual
// tile nt + t is V tile t (nt = ceil(len / KT)) -- the order its producer warp streams them in.  The kernel starts
// under the preceding GEMM (programmatic dependent launch) while the HBM is idle, but its shared-memory ring only
// holds the first 4-6 tiles; the producer therefore also pulls the next `pf_tiles` tiles into L2 with
// cp.async.bulk.prefetch.L2 (UBLKPF) and the later bulk copies hit L2.  Nothing but cache state changes (bit-identical
// results: tests/test_gpu_parity.py::test_kv_l2_prefetch_is_value_neutral).  Measured (profiles/r02_call63_*): 16 tiles
// -1.6 % per batch; the same prefetch issued earlier, from the GEMMs of the previous layer, +0.8 .. +3.4 % (the
// prefetched rows compete with the decoder weights for L2), a persisting-L2 window over the weights 0 .. +1.2 % --
// both removed again.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void l2_prefetch_bulk(const void* gsrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes) : "memory");
}

struct DecGemmArgs {
  const float* A; int lda;        // [M, K]
  const float* W; int ldw;        // [K, N] row-major
  int M, N, K;
  int norm;                       // 1: scale row m by rsqrt(mean(A[m,:]^2) + eps); needs K == row length
  float eps;
  int epi;
  const float* R; int ldr;
  float* C; int ldc;
  int n_split; void* C1; int kv_fmt; int hm_rows_per_b; int hm_cap; int hm_H; const int* hm_pos;   // KV append (kv_fmt: see kv_dest())
  float* partial;                 // [splits][n_tiles][64*32 + 64] scratch (non-cluster fallback)
  int* counters;                  // [n_tiles], zero on entry, left zero on exit
  // optional second activation source: columns [K0, K) of the virtual A come from A2[:, k - K0] (fused launches
  // multiply the concatenation [o | y] by a precomposed weight block); A2 == nullptr -> single source
  const float* A2; int lda2; int K0;
  // optional: per (row, 32-column tile) sum of squares of the OUTPUT row slice, [M][ssq_ld]; the consumer of the
  // output sums the N/32 partials in order and gets the RMSNorm statistic without re-reading the row
  float* ssq_out; int ssq_ld;
  unsigned long long* trace;      // debug timeline slot (mt3_debug_trace_step) or null: [0] min start, [1] max end (ns,
                                  // %globaltimer); [2..6] clock64 deltas of CTA (0,0) at its phase boundaries
};

__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

constexpr int kDecBM = 64, kDecBN = 32, kDecKC = 64;     // output tile 64 x 32, K chunk per CTA (fallback kernel)
constexpr int kDecTileFloats = kDecBM * kDecBN + kDecBM;   // partial tile + per-row sum of squares

// store 4 consecutive outputs of row m starting at column n (relative to the GEMM's N): plain C, or the head-major
// KV cache (fp32 / fp16)
__device__ __forceinline__ void dec_store4(const DecGemmArgs& p, int m, int n, float4 v) {
  if (n < p.n_split) {
    *reinterpret_cast<float4*>(p.C + (long long)m * p.ldc + n) = v;
    return;
  }
  int d;
  char* row = reinterpret_cast<char*>(p.C1) + kv_dest(m, n - p.n_split, p.hm_rows_per_b, p.hm_cap, p.hm_H, p.hm_pos ? *p.hm_pos : 0, p.kv_fmt, d);
  const float v4[4] = {v.x, v.y, v.z, v.w};
  kv_store<4>(row, p.kv_fmt, d, v4);
}

// Non-cluster fallback.  Each CTA handles ONE K chunk of 64: all of its global loads (8 KB of weights, 16 KB of
// activations) are issued before anything is consumed, then the 64 k-steps run out of shared memory.
__global__ void __launch_bounds__(128)
sgemm_dec_kernel(const DecGemmArgs p) {
  constexpr int BM = kDecBM, BN = kDecBN, KC = kDecKC, NT = 128, APAD = 4;
  __shared__ __align__(16) float As[KC][BM + APAD];      // transposed: [k][m]
  __shared__ __align__(16) float Bs[KC][BN];
  __shared__ float s_ss[BM];
  __shared__ int s_last;

  const int tid = threadIdx.x;
  const int tx = tid % 8, ty = tid / 8;                  // thread tile: rows ty*4.., cols tx*4..
  const int n0 = blockIdx.x * BN;
  const int splits = gridDim.y, ks = blockIdx.y;
  const int kbeg = ks * KC;                              // host guarantees K == splits * KC

  float4 rb[4], ra[8];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int idx = tid + i * NT;                        // 512 float4: [64 k][8 column quads]
    const int kr = idx >> 3, nq = idx & 7;
    rb[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n0 + nq * 4 < p.N) rb[i] = __ldg(reinterpret_cast<const float4*>(p.W + (long long)(kbeg + kr) * p.ldw + n0 + nq * 4));
  }
  pdl_wait();
  pdl_trigger();
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int idx = tid + i * NT;                        // 1024 float4: [64 m][16 k quads]
    const int row = idx >> 4, kq = idx & 15;
    ra[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < p.M) ra[i] = *reinterpret_cast<const float4*>(p.A + (long long)row * p.lda + kbeg + kq * 4);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int idx = tid + i * NT;
    *reinterpret_cast<float4*>(&Bs[idx >> 3][(idx & 7) * 4]) = rb[i];
  }
  float ss[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int idx = tid + i * NT;
    const int row = idx >> 4, kq = idx & 15;
    As[kq * 4 + 0][row] = ra[i].x;
    As[kq * 4 + 1][row] = ra[i].y;
    As[kq * 4 + 2][row] = ra[i].z;
    As[kq * 4 + 3][row] = ra[i].w;
    float v = ra[i].x * ra[i].x + ra[i].y * ra[i].y + ra[i].z * ra[i].z + ra[i].w * ra[i].w;
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    ss[i] = v;                                           // sum of squares of row (tid>>4) + 8 i over this K chunk
  }
  __syncthreads();

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
#pragma unroll 16
  for (int k = 0; k < KC; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
    const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
    const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
  }

  const int n_tiles = gridDim.x;
  if (splits > 1) {
    float* mine = p.partial + ((long long)ks * n_tiles + blockIdx.x) * kDecTileFloats;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(mine + (ty * 4 + i) * BN + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    if ((tid & 15) == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) mine[BM * BN + (tid >> 4) + 8 * i] = ss[i];
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      const int ticket = atomicAdd(&p.counters[blockIdx.x], 1);
      s_last = (ticket == splits - 1);
      if (s_last) p.counters[blockIdx.x] = 0;            // re-arm for the next launch
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // fixed-order reduction of all partials (including our own) -> bit-reproducible
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float sst = 0.f;
    for (int s0 = 0; s0 < splits; s0 += 4) {
      float4 v[4][4];
      float sv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {                      // 4 partial tiles in flight per round
        const int s = s0 + u;
        const float* src = p.partial + ((long long)min(s, splits - 1) * n_tiles + blockIdx.x) * kDecTileFloats;
#pragma unroll
        for (int i = 0; i < 4; ++i) v[u][i] = __ldcg(reinterpret_cast<const float4*>(src + (ty * 4 + i) * BN + tx * 4));
        sv[u] = (tid < BM) ? __ldcg(src + BM * BN + tid) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (s0 + u < splits) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            acc[i][0] += v[u][i].x; acc[i][1] += v[u][i].y; acc[i][2] += v[u][i].z; acc[i][3] += v[u][i].w;
          }
          sst += sv[u];
        }
      }
    }
    if (tid < BM) s_ss[tid] = sst;
  } else {
    if ((tid & 15) == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) s_ss[(tid >> 4) + 8 * i] = ss[i];
    }
  }
  __syncthreads();

  // ---- fused epilogue (same set as gemm_simt.cuh) ----
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = ty * 4 + i;
    if (m >= p.M) continue;
    const int n = n0 + tx * 4;
    if (n >= p.N) continue;
    const float rs = p.norm ? 1.0f / sqrtf(s_ss[m] / (float)p.K + p.eps) : 1.f;
    float4 v = make_float4(acc[i][0] * rs, acc[i][1] * rs, acc[i][2] * rs, acc[i][3] * rs);
    if (p.epi == EPI_GATED_GELU) {
      *reinterpret_cast<float2*>(p.C + (long long)m * p.ldc + (n >> 1)) = make_float2(gelu_tanh(v.x) * v.y, gelu_tanh(v.z) * v.w);
      continue;
    }
    if (p.epi == EPI_RESIDUAL) {
      const float4 q = *reinterpret_cast<const float4*>(p.R + (long long)m * p.ldr + n);
      v.x += q.x; v.y += q.y; v.z += q.z; v.w += q.w;
    }
    dec_store4(p, m, n, v);
  }
}

// ---------------------------------------------------------------------------------------------
// Cluster variant (the default on sm_100a): the S (8 or 16) CTAs of one 64 x 32 output tile form a thread-block
// cluster (1, S, 1) and split K.  Each CTA computes the partial tile of its K chunk -- G groups of four warps split
// the chunk once more and are summed through shared memory in group order -- then PUSHES the 64/S rows owned by
// rank r into rank r's shared memory (st.shared::cluster); after ONE cluster barrier every rank sums the S partials
// of its own rows from LOCAL shared memory in rank order (bit-reproducible), applies the fused epilogue and stores.
// No global scratch, no atomics, no second barrier (nobody reads remote memory after the barrier, so a CTA may exit
// as soon as it is done).  The default (MT3_DEC_PIPE=3, below) stages the loads under the multiply and replaces the
// stores + barrier by bulk copies that complete on each receiver's own mbarrier.
//
// Arithmetic: exact fp32 FMA, k ascending inside a group, as packed FFMA2 (ffma2() in common.cuh).  The tensor-core
// variants of round 1 (mma.sync 3xTF32, tcgen05 3xTF32) were parity-green but not faster and live in
// csrc/experiments/ with their measurements.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_map(uint32_t smem_addr, unsigned rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f4(uint32_t addr, float4 v) {
  asm volatile("st.shared::cluster.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_cluster_f1(uint32_t addr, float x) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(addr), "f"(x) : "memory");
}
// local shared memory -> a peer's shared memory (DSMEM) by the bulk-copy engine; completion is counted in bytes on the
// peer's mbarrier (dst and bar: shared::cluster addresses of the same CTA)
__device__ __forceinline__ void bulk_s2c(uint32_t dst, uint32_t src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "r"(src), "r"(bytes), "r"(bar) : "memory");
}
// wait for the bytes sent to this CTA (phase 0 of its exchange mbarrier); cluster-scope acquire: the writers are peers.
// Bounded spin like tc::mbar_wait.
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  do {
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t}"
        : "=r"(ok)
        : "r"(tc::smem_u32(bar)), "r"(parity)
        : "memory");
    if (!ok && ++spins > (1u << 26)) __trap();
  } while (!ok);
}
// cp.async.wait_group takes an immediate: n = groups that may still be pending (0 .. 7)
__device__ __forceinline__ void cp_async_wait_pending(int n) {
  switch (n) {
    case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
    case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
    case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
    case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
    case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
    case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
    case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
    default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
  }
}

constexpr int kDecLDB = kDecBN + 8;            // padded weight rows
constexpr int kDecRedFloats = 8 * 8 * kDecBN;  // [src rank][local rows][32 cols] partials pushed to this CTA (S*R = 64 rows)
template <int KC, int G, int PIPE>
constexpr size_t dec_cluster_smem() {
  return (size_t)(kDecBM * (KC + 4) + KC * kDecLDB + kDecRedFloats + 64 + (G > 1 ? kDecBM * kDecBN : 0)) * sizeof(float) +
         ((PIPE & 2) ? 16 : 0);   // exchange mbarrier
}

// Sum this rank's 64/S rows over the S source ranks (rank order, local shared memory) and apply the fused epilogue:
// RMSNorm row factor, gated-GELU / residual, plain store or head-major KV-cache append.  Threads 0..127; S = 8: 8 rows x
// 16 column pairs, S = 16: 4 rows x 32 single columns (no gated-GELU, whose inputs are column pairs).
template <int S>
__device__ __forceinline__ void dec_reduce_epilogue(const DecGemmArgs& p, const float* Red, const float* Rss, unsigned rank, int n0) {
  constexpr int BN = kDecBN, R = kDecBM / S, CPT = (R * BN) / 128, LPR = BN / CPT;   // rows per rank, columns per thread, lanes per row
  static_assert(CPT == 1 || CPT == 2, "cluster size must be 8 or 16");
  const int tid = threadIdx.x;
  const int rl = tid / LPR, c0 = (tid % LPR) * CPT;
  const int m = (int)rank * R + rl, n = n0 + c0;
  float v[2] = {0.f, 0.f};
  float sst = 0.f;
#pragma unroll
  for (int s = 0; s < S; ++s) {
    if (CPT == 2) {
      const float2 q = *reinterpret_cast<const float2*>(&Red[(s * R + rl) * BN + c0]);
      v[0] += q.x; v[1] += q.y;
    } else {
      v[0] += Red[(s * R + rl) * BN + c0];
    }
    if (p.norm) sst += Rss[s * R + rl];
  }
  const bool valid = m < p.M && n < p.N;
  if (valid) {
    const float rs = p.norm ? 1.0f / sqrtf(sst / (float)p.K + p.eps) : 1.f;
    v[0] *= rs; v[1] *= rs;
    if (CPT == 2 && p.epi == EPI_GATED_GELU) {
      p.C[(long long)m * p.ldc + (n >> 1)] = gelu_tanh(v[0]) * v[1];
    } else {
      if (p.epi == EPI_RESIDUAL) {
        const float* r = p.R + (long long)m * p.ldr + n;
        v[0] += r[0];
        if (CPT == 2) v[1] += r[1];
      }
      if (n < p.n_split) {
        float* dst = p.C + (long long)m * p.ldc + n;
        if (CPT == 2) *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
        else dst[0] = v[0];
      } else {
        int d;
        char* row = reinterpret_cast<char*>(p.C1) + kv_dest(m, n - p.n_split, p.hm_rows_per_b, p.hm_cap, p.hm_H, p.hm_pos ? *p.hm_pos : 0, p.kv_fmt, d);
        kv_store<CPT>(row, p.kv_fmt, d, v);
      }
    }
  }
  if (p.ssq_out) {                      // LPR lanes share a row: fixed butterfly order
    float sq = valid ? fmaf(v[0], v[0], CPT == 2 ? v[1] * v[1] : 0.f) : 0.f;
#pragma unroll
    for (int o = LPR / 2; o >= 1; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((tid % LPR) == 0 && m < p.M) p.ssq_out[(long long)m * p.ssq_ld + n0 / BN] = sq;
  }
}

// PIPE (MT3_DEC_PIPE, bitmask; 0 = the plain sequence above).  Neither bit changes an FMA, its operands or its order:
//  bit 0, staged loads: the activations arrive in cp.async groups of kDecStageK k-steps (one trip of the multiply loop);
//         the multiply of stage s waits for stage s only, so the FMAs start while later stages are still in flight.
//         The weights are issued before the PDL wait as in the plain form and travel in the first group.
//  bit 1, bulk exchange: each CTA writes its partial tile (and per-row sums of squares) row-major into its own, now dead,
//         activation buffer and sends rank r's rows with ONE cp.async.bulk shared::cta -> shared::cluster copy per peer,
//         completing on the receiver's mbarrier; a rank reduces as soon as ITS bytes have landed -- no second cluster
//         barrier, so ranks no longer wait for the slowest peer to finish receiving.
// Measured on a B200 (1000 W limit), whole 64-segment batch, one process (profiles/r03_call1_ab_dec_pipe.txt): 0 454.6,
// 1 432.4, 2 442.6, 3 429.7 ms -- both bits win, and together most; 3 is the default.
constexpr int kDecStageK = 16;

template <int KC, bool TRACE, int S, int G, int PIPE>
__device__ __forceinline__ void dec_cluster_body(const DecGemmArgs& p, const int tile_x) {
  constexpr int BM = kDecBM, BN = kDecBN, NT = 128 * G, LDA = KC + 4, LDB = kDecLDB;
  constexpr int R = BM / S;                   // rows of the tile each rank owns (8 for clusters of 8, 4 for clusters of 16)
  constexpr int KG = KC / G;                  // k-steps per warp group
  static_assert(KG % 4 == 0 && (KC / (2 * G)) % 4 == 0, "K chunk must split into float4 pieces per group / per ssq thread");
  constexpr bool STAGED = (PIPE & 1) != 0, BULK = (PIPE & 2) != 0;
  constexpr int NS = KC / kDecStageK;         // load stages
  static_assert(!STAGED || (G == 1 && KC % kDecStageK == 0 && NS <= 8), "staged loads: one warp group, K chunk of 16 k-step stages");
  static_assert(!BULK || BM * (BN + 1) <= BM * LDA, "bulk exchange: the partial tile + sums of squares are staged in the activation buffer");
  extern __shared__ __align__(16) float dsm[];
  float* As = dsm;                            // [BM][LDA] activations, row-major
  float* Bs = As + BM * LDA;                  // [KC][LDB] weights
  float* Red = Bs + KC * LDB;                 // [S src][R rows][BN] partial tiles of MY rows (written by all ranks)
  float* Rss = Red + kDecRedFloats;           // [S src][R rows] partial sums of squares of my rows
  float* Part = Rss + 64;                     // [BM][BN] partial tile of warp group 1 (G == 2)
  uint64_t* xbar = reinterpret_cast<uint64_t*>(Part + (G > 1 ? BM * BN : 0));   // exchange mbarrier (bulk exchange)

  unsigned rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  const int tid = threadIdx.x;
  const int grp = tid >> 7, t128 = tid & 127;
  const int n0 = tile_x * BN;
  const int kbeg = blockIdx.y * KC;
  const bool tr = TRACE && p.trace != nullptr && tid == 0;
  const bool tr0 = tr && tile_x == 0 && blockIdx.y == 0;
  long long c0 = 0;
  if (tr) {
    atomicMin(p.trace, gtime_ns());
    c0 = clock64();
    if (tile_x == 0) {
      unsigned smid;
      asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
      if (blockIdx.y < 8) p.trace[8 + blockIdx.y] = smid;
    }
  }
  // bulk exchange: the mbarrier the peers' copies complete on, armed for all S * (R rows + R sums of squares) words
  // before the cluster arrive below, which publishes it (fence.mbarrier_init) to the peers
  if constexpr (BULK) {
    if (tid == 0) {
      tc::mbar_init(xbar, 1);
      tc::mbar_arrive_expect_tx(xbar, (uint32_t)(S * R * (BN + 1) * 4));
      tc::fence_barrier_init();
    }
  }
  // "I am running": peers may write into my shared memory once every CTA of the cluster has arrived here
  asm volatile("barrier.cluster.arrive.relaxed.aligned;" ::: "memory");

  // ---- load phase: cp.async (global -> shared, no register staging).  Weights are issued BEFORE the PDL wait (they
  // do not depend on the previous kernel).
  for (int idx = tid; idx < KC * 8; idx += NT) {
    const int kr = idx >> 3, nq = idx & 7;
    const bool ok = n0 + nq * 4 < p.N;
    const float* src = p.W + (long long)(kbeg + kr) * p.ldw + (ok ? n0 + nq * 4 : 0);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(&Bs[kr * LDB + nq * 4])), "l"(src),
                 "r"(ok ? 16 : 0) : "memory");
  }
  pdl_wait();
  pdl_trigger();
  if constexpr (STAGED) {
    // activations in NS commit groups of kDecStageK k-steps (64 rows x 4 float4 each); the multiply waits stage by stage
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      for (int idx = tid; idx < BM * (kDecStageK / 4); idx += NT) {
        const int row = idx / (kDecStageK / 4), kq = s * (kDecStageK / 4) + idx % (kDecStageK / 4);
        const bool ok = row < p.M;
        const int col = kbeg + kq * 4;
        const float* src = (p.A2 != nullptr && col >= p.K0) ? p.A2 + (long long)(ok ? row : 0) * p.lda2 + (col - p.K0)
                                                             : p.A + (long long)(ok ? row : 0) * p.lda + col;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(&As[row * LDA + kq * 4])), "l"(src),
                     "r"(ok ? 16 : 0) : "memory");
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
  } else {
    // all of the CTA's activations in flight at once; one wait
    for (int idx = tid; idx < KC * 16; idx += NT) {
      const int row = idx / (KC / 4), kq = idx % (KC / 4);
      const bool ok = row < p.M;
      const int col = kbeg + kq * 4;
      const float* src = (p.A2 != nullptr && col >= p.K0) ? p.A2 + (long long)(ok ? row : 0) * p.lda2 + (col - p.K0)
                                                           : p.A + (long long)(ok ? row : 0) * p.lda + col;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(tc::smem_u32(&As[row * LDA + kq * 4])), "l"(src),
                   "r"(ok ? 16 : 0) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (tr0) p.trace[2] = (unsigned long long)(clock64() - c0);    // loads landed
  }

  // sum of squares of this CTA's K chunk: 2 G threads per row, each a contiguous piece, fixed butterfly order
  // (staged loads: once the last stage has landed)
  float ss = 0.f;
  auto sum_squares = [&]() {
    if (p.norm) {
      constexpr int PIECE = KC / (2 * G);
      const float* ar = As + (tid / (2 * G)) * LDA + (tid % (2 * G)) * PIECE;
#pragma unroll
      for (int k = 0; k < PIECE; k += 4) {
        const float4 v = *reinterpret_cast<const float4*>(ar + k);
        ss = fmaf(v.x, v.x, ss); ss = fmaf(v.y, v.y, ss); ss = fmaf(v.z, v.z, ss); ss = fmaf(v.w, v.w, ss);
      }
      ss += __shfl_xor_sync(0xffffffffu, ss, 1);
      if (G == 2) ss += __shfl_xor_sync(0xffffffffu, ss, 2);
    }
  };
  if constexpr (!STAGED) sum_squares();

  // ---- multiply: thread tile rows ty + 16 i (i < 4), columns tx*4 .. +3 (two float2 accumulators per row); warp
  // group g covers k in [g KG, (g+1) KG), ascending ----
  const int tx = t128 % 8, ty = t128 / 8;
  float2 acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
  {
    const float* Ag = As + grp * KG;
    const float* Bg = Bs + grp * KG * LDB;
    auto fma4 = [&](int k) {                                        // k-steps k .. k+3
      float4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(&Ag[(ty + 16 * i) * LDA + k]);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) b[kk] = *reinterpret_cast<const float4*>(&Bg[(k + kk) * LDB + tx * 4]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float av[4] = {a[i].x, a[i].y, a[i].z, a[i].w};
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          ffma2(acc[i][0], av[kk], make_float2(b[kk].x, b[kk].y));
          ffma2(acc[i][1], av[kk], make_float2(b[kk].z, b[kk].w));
        }
      }
    };
    if constexpr (STAGED) {
#pragma unroll 1
      for (int s = 0; s < NS; ++s) {                                // one trip per stage, k ascending as below
        cp_async_wait_pending(NS - 1 - s);
        __syncthreads();                                            // rows of As are filled by other threads
        if (tr0 && s == 0) p.trace[2] = (unsigned long long)(clock64() - c0);   // first stage landed
#pragma unroll
        for (int k = s * kDecStageK; k < (s + 1) * kDecStageK; k += 4) fma4(k);
      }
      sum_squares();
    } else {
#pragma unroll 4
      for (int k = 0; k < KG; k += 4) fma4(k);
    }
  }
  if (G == 2) {                                                     // group 1 -> shared memory -> added by group 0
    if (grp == 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(&Part[(ty + 16 * i) * BN + tx * 4]) = make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
    }
    __syncthreads();
    if (grp == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 q = *reinterpret_cast<const float4*>(&Part[(ty + 16 * i) * BN + tx * 4]);
        acc[i][0].x += q.x; acc[i][0].y += q.y; acc[i][1].x += q.z; acc[i][1].y += q.w;
      }
    }
  }
  if (tr0) p.trace[3] = (unsigned long long)(clock64() - c0);      // multiply done
  asm volatile("barrier.cluster.wait.aligned;" ::: "memory");      // every peer is running

  const uint32_t red_base = tc::smem_u32(Red) + rank * (R * BN * 4);     // my slot [rank][..] in the owner's Red
  const uint32_t rss_base = tc::smem_u32(Rss) + rank * (R * 4);
  if constexpr (BULK) {
    // partial tile [BM][BN] row-major, then the BM row sums of squares, over the activation buffer: rank r's rows are
    // one contiguous R * BN * 4-byte slice
    float* Xs = As;
    __syncthreads();                                                // every read of As (multiply, sums of squares) is done
    if (grp == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        *reinterpret_cast<float4*>(&Xs[(ty + 16 * i) * BN + tx * 4]) = make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
    }
    if ((tid % (2 * G)) == 0) Xs[BM * BN + tid / (2 * G)] = ss;
    tc::fence_proxy_async();                                        // generic-proxy stores -> the bulk copies read them
    __syncthreads();
    if (tid < S) {                                                  // thread r sends rank r its rows
      const uint32_t bar = cluster_map(tc::smem_u32(xbar), (unsigned)tid);
      bulk_s2c(cluster_map(red_base, (unsigned)tid), tc::smem_u32(Xs + tid * R * BN), (uint32_t)(R * BN * 4), bar);
      bulk_s2c(cluster_map(rss_base, (unsigned)tid), tc::smem_u32(Xs + BM * BN + tid * R), (uint32_t)(R * 4), bar);
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    if (grp == 0) mbar_wait_cluster(xbar, 0);                       // my rows from all S ranks have landed
  } else {
    if (grp == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {                                // row ty + 16 i -> owner rank, local row
        const int row = ty + 16 * i;
        st_cluster_f4(cluster_map(red_base + (uint32_t)(((row % R) * BN + tx * 4) * 4), (unsigned)(row / R)),
                      make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y));
      }
    }
    if (p.norm && (tid % (2 * G)) == 0) {
      const int row = tid / (2 * G);
      st_cluster_f1(cluster_map(rss_base + (uint32_t)((row % R) * 4), (unsigned)(row / R)), ss);
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
  }
  if (tr0) p.trace[4] = (unsigned long long)(clock64() - c0);      // partials exchanged

  if (grp == 0) dec_reduce_epilogue<S>(p, Red, Rss, rank, n0);
  // the CTA (and its staging buffer) must outlive the bulk copies' reads of it
  if (BULK && tid < S) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  if (tr) {
    if (tr0) p.trace[5] = (unsigned long long)(clock64() - c0);    // reduce + epilogue stores issued
    atomicMax(p.trace + 1, gtime_ns());
  }
}

template <int KC, bool TRACE, int S, int G, int PIPE>
__global__ void __launch_bounds__(128 * G)
sgemm_dec_cluster_kernel(const DecGemmArgs p) {
  dec_cluster_body<KC, TRACE, S, G, PIPE>(p, (int)blockIdx.x);
}

// Two independent GEMMs that read the same inputs in ONE launch (column tiles [0, tiles0) belong to p0, the rest to
// p1): used for  y' = y + o.Wo  together with  q_raw = [o | y].[Wo.Wq ; Wq]  (the out-projection folded into the
// next projection with a precomposed weight block), which removes a kernel from the dependency chain.
template <int KC0, int KC1, bool TRACE, int G, int PIPE>
__global__ void __launch_bounds__(128 * G)
sgemm_dec_cluster2_kernel(const DecGemmArgs p0, const DecGemmArgs p1, const int tiles0) {
  if ((int)blockIdx.x < tiles0) dec_cluster_body<KC0, TRACE, 8, G, PIPE>(p0, (int)blockIdx.x);
  else dec_cluster_body<KC1, TRACE, 8, G, PIPE>(p1, (int)blockIdx.x - tiles0);
}

// One warp group (128 threads) per CTA.  The body is also written for G = 2 groups that split the CTA's K chunk once
// more and are summed through shared memory; measured on a B200 that is slower (437.8 vs 429.1 ms per batch,
// profiles/r02_call1_*): the multiply loop is bound by shared-memory bandwidth (8 LDS.128 per 64 FMAs with 4 x 4
// register tiles), not by issue latency, so more warps only add the combine step.  For the same reason FFMA2 is not
// faster than scalar FFMA here.  (The staged loads of MT3_DEC_PIPE bit 0 are written for one group only.)
constexpr int kDecGroups = 1;

// runtime MT3_DEC_PIPE bits -> the kernel instantiation
#define MT3_DEC_PIPE_DISPATCH(pipe, CALL) \
  switch ((pipe) & 3) {                   \
    case 0: return CALL(0);               \
    case 1: return CALL(1);               \
    case 2: return CALL(2);               \
    default: return CALL(3);              \
  }

template <int KC0, int KC1, int G, int PIPE>
inline int launch_dec_gemm_cluster2_g(const DecGemmArgs& a0, const DecGemmArgs& a1, cudaStream_t s, bool pdl) {
  constexpr size_t smem = dec_cluster_smem<(KC0 > KC1 ? KC0 : KC1), G, PIPE>();
  static bool attr_done = false;
  if (!attr_done) {
    MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster2_kernel<KC0, KC1, false, G, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster2_kernel<KC0, KC1, true, G, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_done = true;
  }
  const int tiles0 = a0.N / kDecBN, tiles1 = a1.N / kDecBN;
  if (a0.trace)
    MT3_CUDA_CHECK(launch_kernel_cluster(sgemm_dec_cluster2_kernel<KC0, KC1, true, G, PIPE>, dim3(tiles0 + tiles1, 8), dim3(128 * G), smem, s,
                                         pdl, 8u, a0, a1, tiles0));
  else
    MT3_CUDA_CHECK(launch_kernel_cluster(sgemm_dec_cluster2_kernel<KC0, KC1, false, G, PIPE>, dim3(tiles0 + tiles1, 8), dim3(128 * G), smem, s,
                                         pdl, 8u, a0, a1, tiles0));
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

// the mt3 shapes: K = 384 (out-projection) and K = 384 + 512 (precomposed query block)
inline int launch_dec_gemm_out_q(const DecGemmArgs& a0, const DecGemmArgs& a1, cudaStream_t s, bool pdl, int pipe) {
  if (a0.M > kDecBM || a1.M > kDecBM || a0.K != 8 * 48 || a1.K != 8 * 112 || a0.N % kDecBN != 0 || a1.N % kDecBN != 0)
    return MT3_ERR_UNSUPPORTED;
#define MT3_CALL(P) launch_dec_gemm_cluster2_g<48, 112, kDecGroups, P>(a0, a1, s, pdl)
  MT3_DEC_PIPE_DISPATCH(pipe, MT3_CALL)
#undef MT3_CALL
}

template <int KC, int S, int G, int PIPE>
inline int launch_dec_gemm_cluster_kc(const DecGemmArgs& a, cudaStream_t s, bool pdl) {
  constexpr size_t smem = dec_cluster_smem<KC, G, PIPE>();
  static bool attr_done = false;
  if (!attr_done) {
    MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster_kernel<KC, false, S, G, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster_kernel<KC, true, S, G, PIPE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (S > 8) {
      MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster_kernel<KC, false, S, G, PIPE>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      MT3_CUDA_CHECK(cudaFuncSetAttribute(sgemm_dec_cluster_kernel<KC, true, S, G, PIPE>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    }
    attr_done = true;
  }
  if (a.trace)
    MT3_CUDA_CHECK(launch_kernel_cluster(sgemm_dec_cluster_kernel<KC, true, S, G, PIPE>, dim3(cdiv(a.N, kDecBN), S), dim3(128 * G), smem, s, pdl, (unsigned)S, a));
  else
    MT3_CUDA_CHECK(launch_kernel_cluster(sgemm_dec_cluster_kernel<KC, false, S, G, PIPE>, dim3(cdiv(a.N, kDecBN), S), dim3(128 * G), smem, s, pdl, (unsigned)S, a));
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

template <int KC, int S, int G>
inline int launch_dec_gemm_cluster_p(const DecGemmArgs& a, cudaStream_t s, bool pdl, int pipe) {
#define MT3_CALL(P) launch_dec_gemm_cluster_kc<KC, S, G, P>(a, s, pdl)
  MT3_DEC_PIPE_DISPATCH(pipe, MT3_CALL)
#undef MT3_CALL
}

template <int G>
inline int launch_dec_gemm_cluster_g(const DecGemmArgs& a, cudaStream_t s, bool pdl, int pipe) {
  // the long-K, narrow-N GEMM (MLP out: K = 1024, N = 512) has only N/32 x 8 = 128 CTAs at cluster size 8: a
  // cluster of 16 halves every CTA's K chunk and fills the machine
  if ( a.K == 1024 && a.epi != EPI_GATED_GELU && a.N <= 512) return launch_dec_gemm_cluster_p<64, 16, G>(a, s, pdl, pipe);
  switch (a.K / 8) {
    case 48: return launch_dec_gemm_cluster_p<48, 8, G>(a, s, pdl, pipe);
    case 64: return launch_dec_gemm_cluster_p<64, 8, G>(a, s, pdl, pipe);
    case 128: return launch_dec_gemm_cluster_p<128, 8, G>(a, s, pdl, pipe);
    default: return MT3_ERR_UNSUPPORTED;
  }
}

// Returns MT3_ERR_UNSUPPORTED (without launching) when K does not split into 8 chunks of 48/64/128.
// pipe: MT3_DEC_PIPE bits (dec_cluster_body).
inline int launch_dec_gemm_cluster(const DecGemmArgs& a, cudaStream_t s, bool pdl, int pipe) {
  if (a.M > kDecBM || a.N % 4 != 0 || a.lda % 4 != 0 || a.ldw % 4 != 0 || a.n_split % 4 != 0 || a.K % 8 != 0) return MT3_ERR_UNSUPPORTED;
  return launch_dec_gemm_cluster_g<kDecGroups>(a, s, pdl, pipe);
}

inline int launch_dec_gemm(const DecGemmArgs& a, cudaStream_t s, bool pdl = false) {
  MT3_REQUIRE(a.M <= kDecBM, MT3_ERR_UNSUPPORTED, "decode gemm: M=%d > %d rows", a.M, kDecBM);
  MT3_REQUIRE(a.K % kDecKC == 0 && a.K / kDecKC <= 16 && a.N % 4 == 0 && a.lda % 4 == 0 && a.ldw % 4 == 0 && a.n_split % 4 == 0,
              MT3_ERR_UNSUPPORTED, "decode gemm: K=%d must be a multiple of %d (at most 16 chunks); N=%d", a.K, kDecKC, a.N);
  MT3_REQUIRE(a.A2 == nullptr, MT3_ERR_UNSUPPORTED, "decode gemm: the two-source form needs the cluster kernel");
  MT3_CUDA_CHECK(launch_kernel(sgemm_dec_kernel, dim3(cdiv(a.N, kDecBN), a.K / kDecKC), dim3(128), 0, s, pdl, a));
  MT3_LAUNCH_CHECK();
  return MT3_OK;
}

// ---------------------------------------------------------------------------------------------
// Decode attention over head-major K/V, bulk-copy pipelined.  FMT is the row format (kv_dest()): 0 = fp32 rows
// (256 B, 32 keys per 8 KB tile, 6 stages); 1 = fp16 rows (128 B, 64 keys per 8 KB tile, 6 stages); 2 = p24 rows
// (192 B, 64 keys per 12 KB tile, 4 stages).  Rows are widened to fp32 on the way into the FMAs.
// ---------------------------------------------------------------------------------------------
constexpr int kAttRingBytes = 48 * 1024;
constexpr int kAttThreads = 160;                 // 4 consumer warps + 1 producer warp

// element e (0..7) of a p24 chunk: hi = four 32-bit words holding eight u16, lo = two words holding eight u8
__device__ __forceinline__ float p24_elt(const uint4& hi, const uint2& lo, int e) {
  const uint32_t h = e < 2 ? hi.x : (e < 4 ? hi.y : (e < 6 ? hi.z : hi.w));
  const uint32_t l = e < 4 ? lo.x : lo.y;
  const uint32_t lb = 4u + (uint32_t)(e & 3);                              // byte of l (second operand: indices 4..7)
  const uint32_t sel = (e & 1) ? (0x3200u | (lb << 4) | lb) : (0x1000u | (lb << 4) | lb);
  return __uint_as_float(__byte_perm(h, l, sel));
}

// K/V rows are read once per step and are 10x the size of L2: stream them with an evict-first policy so
// that the 104 MB of decoder weights (re-read every step) stay L2-resident.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               :
               : "r"(tc::smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(tc::smem_u32(bar)),
                 "l"(policy)
               : "memory");
}

inline size_t dec_attention_smem(int max_len) {
  return (size_t)kAttRingBytes + (size_t)(4 * ((max_len + 3) & ~3) + 16 * 64 + 64) * sizeof(float) + 2 * 6 * 8 + 64;
}

// q [B, ldq], head h at column q_off + h*64.  kv: head-major [b][2][H][cap] rows of format FMT.  out [B, ldo].
// len = (len_ptr ? *len_ptr : 0) + len_add.
template <int FMT, bool TRACE>
__global__ void __launch_bounds__(kAttThreads)
dec_attention_bulk_kernel(const float* __restrict__ q, int ldq, int q_off, const void* __restrict__ kv_raw, int H, int cap,
                          const int* __restrict__ len_ptr, int len_add, int max_len, float* __restrict__ out, int ldo,
                          const float* __restrict__ q_ssq, int q_ssq_n, int q_ssq_ld, float q_dim, float q_eps,
                          unsigned long long* trace, int pf_tiles) {
  constexpr bool HALF = FMT == 1, P24 = FMT == 2;
  constexpr int KT = FMT == 0 ? 32 : 64;                         // keys per tile
  constexpr int ROWB = FMT == 0 ? 256 : (FMT == 1 ? 128 : 192);  // bytes per key row
  constexpr int kAttTileBytes = KT * ROWB;                       // 8 KB / 8 KB / 12 KB
  constexpr int kAttStages = kAttRingBytes / kAttTileBytes;      // 6 / 6 / 4
  extern __shared__ __align__(128) unsigned char sm_raw[];
  const int ml4 = (max_len + 3) & ~3;
  unsigned char* ring = sm_raw;                                  // [stages][tile]
  float* sP = reinterpret_cast<float*>(ring + kAttStages * kAttTileBytes);   // [4][ml4]: per-warp partial scores; row 0 becomes P
  float* sRed = sP + 4 * ml4;                                    // [16][64]
  float* sQ = sRed + 16 * 64;                                    // [64] the (scaled) query
  uint64_t* full = reinterpret_cast<uint64_t*>(sQ + 64);         // [stages]
  uint64_t* empty = full + 6;
  __shared__ float s_stat[8];

  const int h = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int len = (len_ptr ? *len_ptr : 0) + len_add;
  const int nt = (len + KT - 1) / KT;
  const unsigned char* kbase = reinterpret_cast<const unsigned char*>(kv_raw) + (((long long)b * 2 + 0) * H + h) * (long long)cap * ROWB;
  const unsigned char* vbase = reinterpret_cast<const unsigned char*>(kv_raw) + (((long long)b * 2 + 1) * H + h) * (long long)cap * ROWB;
  const bool tr = TRACE && trace != nullptr && tid == 0;
  const bool tr0 = tr && blockIdx.x == 0 && blockIdx.y == 0;
  long long c0 = 0;
  if (tr) {
    atomicMin(trace, gtime_ns());
    c0 = clock64();
  }

  if (tid == 0) {
    for (int s = 0; s < kAttStages; ++s) {
      tc::mbar_init(&full[s], 1);
      tc::mbar_init(&empty[s], 4);
    }
    tc::fence_barrier_init();
  }
  __syncthreads();

  if (warp == 4) {
    // ---- producer: K tiles 0..nt-1, then V tiles 0..nt-1 ----
    // self-attention (len_ptr set): every cache row but the newest (tile nt-1) was written by earlier steps, so those
    // tiles are streamed before the PDL wait and only the last tile is held back until the QKV GEMM has completed;
    // the hoisted cross K/V is independent of every decode-step kernel -> streamed right away.
    pdl_trigger();
    if (lane == 0) {
      const uint64_t policy = l2_evict_first_policy();
      bool waited = len_ptr == nullptr;
      // L2 prefetch of the pf_tiles virtual tiles that follow the ring's: requested once, AFTER the ring's own loads are
      // in flight and before this warp first blocks (on a ring slot, or on the PDL wait when the cache is still short)
      bool prefetched = pf_tiles <= 0;
      for (int j = 0; j < 2 * nt; ++j) {
        const int s = j % kAttStages;
        const uint32_t ph = (j / kAttStages) & 1;
        const int t = j < nt ? j : j - nt;
        if (!prefetched && (j >= kAttStages || (!waited && t == nt - 1))) {
          for (int jj = max(kAttStages, j); jj < min(kAttStages + pf_tiles, 2 * nt); ++jj) {
            const int tt = jj < nt ? jj : jj - nt;
            l2_prefetch_bulk((jj < nt ? kbase : vbase) + (long long)tt * kAttTileBytes, (uint32_t)(min(KT, len - tt * KT) * ROWB));
          }
          prefetched = true;
        }
        if (!waited && t == nt - 1) {
          pdl_wait();
          waited = true;
        }
        tc::mbar_wait(&empty[s], ph ^ 1);
        const int keys = min(KT, len - t * KT);
        const uint32_t bytes = (uint32_t)keys * ROWB;
        const unsigned char* src = (j < nt ? kbase : vbase) + (long long)t * kAttTileBytes;
        tc::mbar_arrive_expect_tx(&full[s], bytes);
        bulk_g2s(ring + s * kAttTileBytes, src, bytes, &full[s], policy);
      }
    }
    return;
  }

  // ---- consumers (128 threads) ----
  pdl_wait();                                                    // q comes from the preceding GEMM
  pdl_trigger();
  if (tid < 16) {
    float4 q4 = *reinterpret_cast<const float4*>(q + (long long)b * ldq + q_off + h * 64 + tid * 4);
    if (q_ssq) {
      // q arrives un-normalised from a fused projection: scale by rsqrt(mean(y^2) + eps) of its input row, whose sum
      // of squares the producing GEMM left as q_ssq_n per-tile partials (summed in order)
      float ssq = 0.f;
      for (int i = 0; i < q_ssq_n; ++i) ssq += __ldg(q_ssq + (long long)b * q_ssq_ld + i);
      const float rs = 1.0f / sqrtf(ssq / q_dim + q_eps);
      q4.x *= rs; q4.y *= rs; q4.z *= rs; q4.w *= rs;
    }
    reinterpret_cast<float4*>(sQ)[tid] = q4;
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
  // pass 1: scores, no cross-lane traffic.  Lane <-> key of the tile; a warp covers four 16-byte chunks of the key's
  // row, rotated by the lane so that the eight lanes of a quarter-warp hit eight distinct bank groups (rows are
  // bank-aligned).  fp32 rows (16 chunks): warp w covers chunks 4w..4w+3 of keys 0..31, four per-warp partial dot
  // products per key.  fp16 rows (8 chunks of 8 dims): warp w covers chunk half w>>1 of keys 32 (w&1) + lane, two
  // partials per key.  The partials are added in fixed order by the softmax pass.
  {
    // the chunks a lane reads do not depend on the tile: its slice of q lives in registers
    const float4* q4s = reinterpret_cast<const float4*>(sQ);
    float4 qa[4], qb[4];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      if (HALF || P24) {
        const int c = (4 * (warp >> 1) + jj + (lane & 7)) & 7;
        qa[jj] = q4s[2 * c];
        qb[jj] = q4s[2 * c + 1];
      } else {
        qa[jj] = q4s[(4 * warp + jj + (lane & 7)) & 15];
      }
    }
    for (int j = 0; j < nt; ++j) {
      const int s = j % kAttStages;
      tc::mbar_wait(&full[s], (j / kAttStages) & 1);
      if (tr0 && j == 0) trace[2] = (unsigned long long)(clock64() - c0);      // first K tile landed
      const int k0 = j * KT;
      float d = 0.f;
      if (HALF) {
        const int key = (warp & 1) * 32 + lane;
        const uint4* row = reinterpret_cast<const uint4*>(ring + s * kAttTileBytes + key * ROWB);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int c = (4 * (warp >> 1) + jj + (lane & 7)) & 7;
          const uint4 kx = row[c];
          const float2 k01 = __half22float2(*reinterpret_cast<const __half2*>(&kx.x));
          const float2 k23 = __half22float2(*reinterpret_cast<const __half2*>(&kx.y));
          const float2 k45 = __half22float2(*reinterpret_cast<const __half2*>(&kx.z));
          const float2 k67 = __half22float2(*reinterpret_cast<const __half2*>(&kx.w));
          d = fmaf(qa[jj].x, k01.x, d); d = fmaf(qa[jj].y, k01.y, d); d = fmaf(qa[jj].z, k23.x, d); d = fmaf(qa[jj].w, k23.y, d);
          d = fmaf(qb[jj].x, k45.x, d); d = fmaf(qb[jj].y, k45.y, d); d = fmaf(qb[jj].z, k67.x, d); d = fmaf(qb[jj].w, k67.y, d);
        }
        if (k0 + key < len) sP[(warp >> 1) * ml4 + k0 + key] = d;
      } else if (P24) {
        const int key = (warp & 1) * 32 + lane;
        const unsigned char* row = ring + s * kAttTileBytes + key * ROWB;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int c = (4 * (warp >> 1) + jj + (lane & 7)) & 7;
          const uint4 hi = *reinterpret_cast<const uint4*>(row + c * 16);
          const uint2 lo = *reinterpret_cast<const uint2*>(row + 128 + c * 8);
          d = fmaf(qa[jj].x, p24_elt(hi, lo, 0), d); d = fmaf(qa[jj].y, p24_elt(hi, lo, 1), d);
          d = fmaf(qa[jj].z, p24_elt(hi, lo, 2), d); d = fmaf(qa[jj].w, p24_elt(hi, lo, 3), d);
          d = fmaf(qb[jj].x, p24_elt(hi, lo, 4), d); d = fmaf(qb[jj].y, p24_elt(hi, lo, 5), d);
          d = fmaf(qb[jj].z, p24_elt(hi, lo, 6), d); d = fmaf(qb[jj].w, p24_elt(hi, lo, 7), d);
        }
        if (k0 + key < len) sP[(warp >> 1) * ml4 + k0 + key] = d;
      } else {
        const float4* row = reinterpret_cast<const float4*>(ring + s * kAttTileBytes + lane * ROWB);
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const float4 kx = row[(4 * warp + jj + (lane & 7)) & 15];
          d = fmaf(qa[jj].x, kx.x, d); d = fmaf(qa[jj].y, kx.y, d); d = fmaf(qa[jj].z, kx.z, d); d = fmaf(qa[jj].w, kx.w, d);
        }
        if (k0 + lane < len) sP[warp * ml4 + k0 + lane] = d;
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&empty[s]);
    }
  }
  if (tr0) trace[3] = (unsigned long long)(clock64() - c0);       // pass 1 (K tiles) consumed
  asm volatile("bar.sync 1, 128;" ::: "memory");                // all partial rows are complete
  float lmax = -INFINITY;
  for (int k = tid; k < len; k += 128) {
    const float sc = (HALF || P24) ? sP[k] + sP[ml4 + k] : ((sP[k] + sP[ml4 + k]) + sP[2 * ml4 + k]) + sP[3 * ml4 + k];
    sP[k] = sc;
    lmax = fmaxf(lmax, sc);
  }
  lmax = warp_max(lmax);
  if (lane == 0) s_stat[warp] = lmax;
  asm volatile("bar.sync 1, 128;" ::: "memory");
  const float mx = fmaxf(fmaxf(s_stat[0], s_stat[1]), fmaxf(s_stat[2], s_stat[3]));
  float lsum = 0.f;
  for (int k = tid; k < len; k += 128) {
    const float e = expf(sP[k] - mx);
    sP[k] = e;
    lsum += e;
  }
  lsum = warp_sum(lsum);
  if (lane == 0) s_stat[4 + warp] = lsum;
  asm volatile("bar.sync 1, 128;" ::: "memory");
  const float inv = 1.0f / (s_stat[4] + s_stat[5] + s_stat[6] + s_stat[7]);
  if (tr0) trace[4] = (unsigned long long)(clock64() - c0);       // softmax done

  // pass 2: O = P V.  fp32: thread -> key group tid / 16 (8 groups) x 4 dims (tid % 16); fp16: key group tid / 8
  // (16 groups) x 8 dims (tid % 8, one 16-byte chunk of the row)
  constexpr int NG = FMT == 0 ? 8 : 16;
  if (HALF || P24) {
    const int kg = tid >> 3, d8 = tid & 7;
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
    for (int j = nt; j < 2 * nt; ++j) {
      const int s = j % kAttStages;
      tc::mbar_wait(&full[s], (j / kAttStages) & 1);
      const unsigned char* tile = ring + s * kAttTileBytes;
      const int k0 = (j - nt) * KT;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kk = kg + i * 16;
        if (k0 + kk < len) {
          const float pk = sP[k0 + kk];
          const uint4 vx = *reinterpret_cast<const uint4*>(tile + kk * ROWB + d8 * 16);
          float2 v01, v23, v45, v67;
          if (P24) {
            const uint2 lo = *reinterpret_cast<const uint2*>(tile + kk * ROWB + 128 + d8 * 8);
            v01 = make_float2(p24_elt(vx, lo, 0), p24_elt(vx, lo, 1)); v23 = make_float2(p24_elt(vx, lo, 2), p24_elt(vx, lo, 3));
            v45 = make_float2(p24_elt(vx, lo, 4), p24_elt(vx, lo, 5)); v67 = make_float2(p24_elt(vx, lo, 6), p24_elt(vx, lo, 7));
          } else {
            v01 = __half22float2(*reinterpret_cast<const __half2*>(&vx.x));
            v23 = __half22float2(*reinterpret_cast<const __half2*>(&vx.y));
            v45 = __half22float2(*reinterpret_cast<const __half2*>(&vx.z));
            v67 = __half22float2(*reinterpret_cast<const __half2*>(&vx.w));
          }
          acc[0] = fmaf(pk, v01.x, acc[0]); acc[1] = fmaf(pk, v01.y, acc[1]);
          acc[2] = fmaf(pk, v23.x, acc[2]); acc[3] = fmaf(pk, v23.y, acc[3]);
          acc[4] = fmaf(pk, v45.x, acc[4]); acc[5] = fmaf(pk, v45.y, acc[5]);
          acc[6] = fmaf(pk, v67.x, acc[6]); acc[7] = fmaf(pk, v67.y, acc[7]);
        }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&empty[s]);
    }
    if (tr0) trace[5] = (unsigned long long)(clock64() - c0);     // pass 2 (V tiles) consumed
    *reinterpret_cast<float4*>(sRed + kg * 64 + d8 * 8) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    *reinterpret_cast<float4*>(sRed + kg * 64 + d8 * 8 + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
  } else {
    const int kg = tid >> 4, d4 = tid & 15;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = nt; j < 2 * nt; ++j) {
      const int s = j % kAttStages;
      tc::mbar_wait(&full[s], (j / kAttStages) & 1);
      const float* tile = reinterpret_cast<const float*>(ring + s * kAttTileBytes);
      const int k0 = (j - nt) * KT;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kk = kg + i * 8;
        if (k0 + kk < len) {
          const float pk = sP[k0 + kk];
          const float4 v = *reinterpret_cast<const float4*>(tile + kk * 64 + d4 * 4);
          acc.x = fmaf(pk, v.x, acc.x); acc.y = fmaf(pk, v.y, acc.y);
          acc.z = fmaf(pk, v.z, acc.z); acc.w = fmaf(pk, v.w, acc.w);
        }
      }
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(&empty[s]);
    }
    if (tr0) trace[5] = (unsigned long long)(clock64() - c0);     // pass 2 (V tiles) consumed
    *reinterpret_cast<float4*>(sRed + kg * 64 + d4 * 4) = acc;
  }
  asm volatile("bar.sync 1, 128;" ::: "memory");
  if (tid < 64) {
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < NG; ++g) s += sRed[g * 64 + tid];
    out[(long long)b * ldo + h * 64 + tid] = s * inv;
  }
  if (tr) {
    if (tr0) trace[6] = (unsigned long long)(clock64() - c0);
    atomicMax(trace + 1, gtime_ns());
  }
}

}  // namespace mt3
