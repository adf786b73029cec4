// gemm_tcgen05.cu -- D[M,N] = epilogue(A[M,K] . W[N,K]^T): the one dense-contraction kernel of the
// engine (every nn.Linear / 1x1 conv / patch-embed / projector / LM head on the FO1 path).
//
// Blackwell-native structure (no wgmma, no mma.sync):
//   * persistent CTAs, one per SM, static round-robin over 128 x BN output tiles;
//   * warp 0  : TMA producer  -- cp.async.bulk.tensor 2-D tiles (128B swizzle) of A and W into a
//               STAGES-deep shared-memory ring, completion on mbarriers (expect_tx);
//   * warp 1  : MMA issuer    -- one elected thread issues tcgen05.mma (kind::f16, bf16 x bf16 -> fp32,
//               UMMA 128 x BN x 16) straight from shared-memory descriptors into TMEM; tcgen05.commit
//               releases ring slots and publishes finished accumulators;
//   * warps 2-5: epilogue     -- tcgen05.ld TMEM -> registers, bias / GELU / SiLU / gated-SiLU /
//               residual fused, bf16 or fp32 stores.  Two TMEM accumulator stages (2 x BN columns) let
//               the epilogue of tile i overlap the main loop of tile i+1.
// Out-of-bounds rows/cols/K are zero-filled by TMA on load and predicated on store, so M, N, K need no
// padding beyond 16-byte row pitches.
#include <cuda.h>

#include <algorithm>
#include <map>
#include <mutex>

#include "kernels.cuh"
#include "ptx.cuh"

namespace fo1 {

constexpr int BM = 128;
constexpr int BK = 64;  // 64 bf16 = 128 B = one swizzle atom row
constexpr int UMMA_K = 16;
constexpr int kGemmThreads = 320;   // warp 0: TMA, warp 1: MMA, warps 2-9: epilogue (two per TMEM lane quarter)
constexpr int kEpiThreads = 256;

struct GemmArgs {
  int M, N, K;
  void* D; long long ldd; int d_dtype;
  const void* bias; int bias_dtype;
  int act;
  const __nv_bfloat16* residual; long long ldr;
  int gated;
  int tiles_m, tiles_n;
  // split-K (skinny problems): work item = (tile, split); partial sums meet in `ws`, the last CTA to arrive on
  // `counters[tile]` reduces them in split order (deterministic) and runs the epilogue
  int ksplit, kb_per_split;
  int coalesce;   // 1: epilogue stages rows through shared memory and writes full 128-byte lines (needs 16-byte aligned D / residual rows)
  int stages;     // ring depth actually used (<= kMaxStages): skinny problems trade the unused A rows for more stages in flight
  int a_stage_bytes, b_stage_bytes;
  int stage_tx;   // bytes one ring stage receives (A box rows x 128 B + BN x 128 B): skinny problems load only the live A rows
  float* ws;
  int* counters;
  // implicit 3x3 / pad 1 / stride 1 convolution over an NHWC map (conv_cpb = C / 64 k-blocks per tap; 0: ordinary GEMM): the A tile of
  // k-block kb is the [Ht][Wt][64] patch of tap kb / conv_cpb, fetched by a 4-D TMA whose out-of-range coordinates read as zero
  int conv_cpb, conv_H, conv_W, conv_Wt;
};

constexpr int kMaxStages = 24;
template <int BN>
struct GemmCfg {
  static constexpr int kStageBytes = (BM * BK + BN * BK) * 2;
  static constexpr int kStages = (BN == 256) ? 4 : (BN == 192 ? 4 : (BN == 128 ? 6 : (BN == 64 ? 8 : 9)));   // sets the smem budget; the ring depth is planned per launch
  static constexpr int kTmemCols = (BN == 192) ? 512 : 2 * BN;   // TMEM allocations are powers of two
  static constexpr int kStagingBytes = 8 * 4096;   // epilogue: 32 rows x 128 B per epilogue warp
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 512 /*barriers*/ + kStagingBytes;
  static_assert(kSmemBytes <= 232448, "exceeds the 227 KB of shared memory a CTA may opt into");
};

__device__ __forceinline__ float load_bias(const void* bias, int dtype, int n) {
  return dtype == FO1_F32 ? __ldg(static_cast<const float*>(bias) + n)
                          : __bfloat162float(__ldg(static_cast<const __nv_bfloat16*>(bias) + n));
}
// v[0..31] += bias[n .. n+31]  (16-byte vector loads when the 32 columns are in range, scalar tail otherwise)
__device__ __forceinline__ void add_bias32(float (&v)[32], const void* bias, int dtype, int n, int n_limit) {
  if (n + 32 <= n_limit) {
    if (dtype == FO1_F32) {
      const float4* b = reinterpret_cast<const float4*>(static_cast<const float*>(bias) + n);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 t = __ldg(b + q);
        v[q * 4] += t.x; v[q * 4 + 1] += t.y; v[q * 4 + 2] += t.z; v[q * 4 + 3] += t.w;
      }
    } else {
      const uint4* b = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(bias) + n);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 t = __ldg(b + q);
        v[q * 8 + 0] += bf16_lo(t.x); v[q * 8 + 1] += bf16_hi(t.x); v[q * 8 + 2] += bf16_lo(t.y); v[q * 8 + 3] += bf16_hi(t.y);
        v[q * 8 + 4] += bf16_lo(t.z); v[q * 8 + 5] += bf16_hi(t.z); v[q * 8 + 6] += bf16_lo(t.w); v[q * 8 + 7] += bf16_hi(t.w);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (n + j < n_limit) v[j] += load_bias(bias, dtype, n + j);
  }
}
__device__ __forceinline__ float apply_act(float x, int act) {
  if (act == FO1_EPI_GELU) return gelu_erf(x);
  if (act == FO1_EPI_SILU) return silu(x);
  return x;
}
// 32 values of one accumulator row: the activation switch is taken once, not per element
__device__ __forceinline__ void apply_act32(float (&v)[32], int act) {
  if (act == FO1_EPI_GELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
  } else if (act == FO1_EPI_SILU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = silu(v[j]);
  }
}

// residual add + store of 32 consecutive output columns of one row
__device__ __forceinline__ void store_row32(const GemmArgs& g, float (&v)[32], int m, int n, int n_limit) {
  const bool full = (n + 32 <= n_limit);
  if (g.residual != nullptr) {
    const __nv_bfloat16* rp = g.residual + (long long)m * g.ldr + n;
    if (full && ((g.ldr & 7) == 0)) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 rv = __ldg(reinterpret_cast<const uint4*>(rp) + q);
        v[q * 8 + 0] += bf16_lo(rv.x); v[q * 8 + 1] += bf16_hi(rv.x);
        v[q * 8 + 2] += bf16_lo(rv.y); v[q * 8 + 3] += bf16_hi(rv.y);
        v[q * 8 + 4] += bf16_lo(rv.z); v[q * 8 + 5] += bf16_hi(rv.z);
        v[q * 8 + 6] += bf16_lo(rv.w); v[q * 8 + 7] += bf16_hi(rv.w);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (n + j < n_limit) v[j] += __bfloat162float(rp[j]);
    }
  }
  if (g.d_dtype == FO1_BF16) {
    __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(g.D) + (long long)m * g.ldd + n;
    if (full && ((g.ldd & 7) == 0)) {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint4 o;
        o.x = pack_bf16(v[q * 8 + 0], v[q * 8 + 1]);
        o.y = pack_bf16(v[q * 8 + 2], v[q * 8 + 3]);
        o.z = pack_bf16(v[q * 8 + 4], v[q * 8 + 5]);
        o.w = pack_bf16(v[q * 8 + 6], v[q * 8 + 7]);
        reinterpret_cast<uint4*>(dp)[q] = o;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (n + j < n_limit) dp[j] = __float2bfloat16_rn(v[j]);
    }
  } else {
    float* dp = static_cast<float*>(g.D) + (long long)m * g.ldd + n;
    if (full && ((g.ldd & 3) == 0)) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        reinterpret_cast<float4*>(dp)[q] = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (n + j < n_limit) dp[j] = v[j];
    }
  }
}


// 4-column variants for the cooperative split-K reduction
__device__ __forceinline__ void add_bias4(float (&v)[4], const void* bias, int dtype, int n, int n_limit) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (n + j < n_limit) v[j] += load_bias(bias, dtype, n + j);
}
__device__ __forceinline__ void store_row4(const GemmArgs& g, float (&v)[4], int m, int n, int n_limit) {
  const bool full = (n + 4 <= n_limit);
  if (g.residual != nullptr) {
    const __nv_bfloat16* rp = g.residual + (long long)m * g.ldr + n;
    if (full && ((g.ldr & 3) == 0)) {
      const uint2 rv = __ldg(reinterpret_cast<const uint2*>(rp));
      v[0] += bf16_lo(rv.x); v[1] += bf16_hi(rv.x); v[2] += bf16_lo(rv.y); v[3] += bf16_hi(rv.y);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < n_limit) v[j] += __bfloat162float(rp[j]);
    }
  }
  if (g.d_dtype == FO1_BF16) {
    __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(g.D) + (long long)m * g.ldd + n;
    if (full && ((g.ldd & 3) == 0)) {
      *reinterpret_cast<uint2*>(dp) = make_uint2(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]));
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < n_limit) dp[j] = __float2bfloat16_rn(v[j]);
    }
  } else {
    float* dp = static_cast<float*>(g.D) + (long long)m * g.ldd + n;
    if (full && ((g.ldd & 3) == 0)) {
      *reinterpret_cast<float4*>(dp) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < n_limit) dp[j] = v[j];
    }
  }
}
// sum of the ksplit parked partials of 4 consecutive columns (fixed order: deterministic), 4 loads in flight
__device__ __forceinline__ void sum_splits4(float (&v)[4], const float* src, long long sstride, int ksplit) {
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  int sp = 0;
  for (; sp + 4 <= ksplit; sp += 4) {
    const float4 t0 = __ldcg(reinterpret_cast<const float4*>(src + (long long)sp * sstride));
    const float4 t1 = __ldcg(reinterpret_cast<const float4*>(src + (long long)(sp + 1) * sstride));
    const float4 t2 = __ldcg(reinterpret_cast<const float4*>(src + (long long)(sp + 2) * sstride));
    const float4 t3 = __ldcg(reinterpret_cast<const float4*>(src + (long long)(sp + 3) * sstride));
    a.x += (t0.x + t1.x) + (t2.x + t3.x); a.y += (t0.y + t1.y) + (t2.y + t3.y);
    a.z += (t0.z + t1.z) + (t2.z + t3.z); a.w += (t0.w + t1.w) + (t2.w + t3.w);
  }
  for (; sp < ksplit; ++sp) {
    const float4 t = __ldcg(reinterpret_cast<const float4*>(src + (long long)sp * sstride));
    a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
  }
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
}


// ---- coalesced epilogue stores -----------------------------------------------------------------------------
// tcgen05.ld hands every thread ONE accumulator row (32 consecutive columns): storing from there makes each warp
// store touch 32 different rows, 16 bytes each -- fine for compute-bound shapes, ruinous for the memory-bound ones
// (DaViT stage 0: M = 1.6 M rows, K = 256 ran at 0.48 TB/s).  Instead each epilogue warp parks its 32 x 128 B block
// in shared memory (16-byte slots XOR-swizzled by row, conflict-free both ways) and writes it back row-contiguously:
// one instruction = 4 rows x 128 B (or 8 rows x 64 B), the residual is read the same way.
__device__ __forceinline__ void stage_put16(uint8_t* stg, int row, int slot, uint4 v) {
  *reinterpret_cast<uint4*>(stg + row * 128 + ((slot ^ (row & 7)) << 4)) = v;
}
__device__ __forceinline__ uint4 stage_get16(const uint8_t* stg, int row, int slot) {
  return *reinterpret_cast<const uint4*>(stg + row * 128 + ((slot ^ (row & 7)) << 4));
}
// park 32 finished values of this thread's row as bf16 (4 slots) or fp32 (8 slots) starting at slot0
__device__ __forceinline__ void stage_row32(uint8_t* stg, int lane, int slot0, const float (&v)[32], bool bf16_out) {
  if (bf16_out) {
#pragma unroll
    for (int q = 0; q < 4; ++q)
      stage_put16(stg, lane, slot0 + q, make_uint4(pack_bf16(v[q * 8], v[q * 8 + 1]), pack_bf16(v[q * 8 + 2], v[q * 8 + 3]),
                                                    pack_bf16(v[q * 8 + 4], v[q * 8 + 5]), pack_bf16(v[q * 8 + 6], v[q * 8 + 7])));
  } else {
#pragma unroll
    for (int q = 0; q < 8; ++q)
      stage_put16(stg, lane, q, make_uint4(__float_as_uint(v[q * 4]), __float_as_uint(v[q * 4 + 1]), __float_as_uint(v[q * 4 + 2]),
                                            __float_as_uint(v[q * 4 + 3])));
  }
}
// write `segs` 16-byte slots per row of the parked block to D[m_base + row][col0 ...] (+ residual), n_limit = valid columns
__device__ __forceinline__ void flush_rows(const GemmArgs& g, const uint8_t* stg, int lane, int segs, int m_base, int col0, int n_limit) {
  __syncwarp();
  const bool bf16_out = g.d_dtype == FO1_BF16;
  const int epp = bf16_out ? 8 : 4;                // elements per 16-byte slot
  const int rows_per_it = 32 / segs;
  const int seg = lane % segs, r0 = lane / segs;
  const int col = col0 + seg * epp;
  if (bf16_out && g.residual != nullptr && col + 8 <= n_limit) {
    // residual fast path: all residual rows of the block are requested first (up to 8 independent 16-byte loads in
    // flight per lane), then added and stored -- a load -> add -> store chain per row left the K <= 2048 GEMMs with a
    // residual at 720-950 TFLOP/s
    uint4 rr[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int m = m_base + it * rows_per_it + r0;
      rr[it] = make_uint4(0u, 0u, 0u, 0u);
      if (it < segs && m < g.M) rr[it] = __ldg(reinterpret_cast<const uint4*>(g.residual + (long long)m * g.ldr + col));
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int row = it * rows_per_it + r0;
      const int m = m_base + row;
      if (it >= segs || m >= g.M) continue;
      uint4 v = stage_get16(stg, row, seg);
      const uint4 r = rr[it];
      v.x = pack_bf16(bf16_lo(v.x) + bf16_lo(r.x), bf16_hi(v.x) + bf16_hi(r.x));
      v.y = pack_bf16(bf16_lo(v.y) + bf16_lo(r.y), bf16_hi(v.y) + bf16_hi(r.y));
      v.z = pack_bf16(bf16_lo(v.z) + bf16_lo(r.z), bf16_hi(v.z) + bf16_hi(r.z));
      v.w = pack_bf16(bf16_lo(v.w) + bf16_lo(r.w), bf16_hi(v.w) + bf16_hi(r.w));
      *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(g.D) + (long long)m * g.ldd + col) = v;
    }
    __syncwarp();
    return;
  }
  for (int it = 0; it < segs; ++it) {               // segs iterations x rows_per_it rows = 32 rows
    const int row = it * rows_per_it + r0;
    const int m = m_base + row;
    if (m >= g.M || col >= n_limit) continue;
    uint4 v = stage_get16(stg, row, seg);
    if (bf16_out) {
      __nv_bfloat16* dp = static_cast<__nv_bfloat16*>(g.D) + (long long)m * g.ldd + col;
      if (col + 8 <= n_limit) {
        if (g.residual != nullptr) {
          const uint4 r = __ldg(reinterpret_cast<const uint4*>(g.residual + (long long)m * g.ldr + col));
          v.x = pack_bf16(bf16_lo(v.x) + bf16_lo(r.x), bf16_hi(v.x) + bf16_hi(r.x));
          v.y = pack_bf16(bf16_lo(v.y) + bf16_lo(r.y), bf16_hi(v.y) + bf16_hi(r.y));
          v.z = pack_bf16(bf16_lo(v.z) + bf16_lo(r.z), bf16_hi(v.z) + bf16_hi(r.z));
          v.w = pack_bf16(bf16_lo(v.w) + bf16_lo(r.w), bf16_hi(v.w) + bf16_hi(r.w));
        }
        *reinterpret_cast<uint4*>(dp) = v;
      } else {
        const uint32_t u[4] = {v.x, v.y, v.z, v.w};
        for (int j = 0; j < 8 && col + j < n_limit; ++j) {
          float x = (j & 1) ? bf16_hi(u[j >> 1]) : bf16_lo(u[j >> 1]);
          if (g.residual != nullptr) x += __bfloat162float(g.residual[(long long)m * g.ldr + col + j]);
          dp[j] = __float2bfloat16_rn(x);
        }
      }
    } else {
      float* dp = static_cast<float*>(g.D) + (long long)m * g.ldd + col;
      float x[4] = {__uint_as_float(v.x), __uint_as_float(v.y), __uint_as_float(v.z), __uint_as_float(v.w)};
      for (int j = 0; j < 4; ++j)
        if (g.residual != nullptr && col + j < n_limit) x[j] += __bfloat162float(g.residual[(long long)m * g.ldr + col + j]);
      if (col + 4 <= n_limit) *reinterpret_cast<float4*>(dp) = make_float4(x[0], x[1], x[2], x[3]);
      else for (int j = 0; j < 4 && col + j < n_limit; ++j) dp[j] = x[j];
    }
  }
  __syncwarp();
}

// Split-K: the last CTA to park its partial reduces the tile.  Kept out of line so that its registers do not weigh
// on the allocation of the main epilogue (the kernel runs at the 168-register cap of 3 warps per SM sub-partition).
template <int BN>
__device__ __noinline__ void splitk_finish(const GemmArgs& g, int tile, int m0, int n0) {
  // all 256 epilogue threads share the tile: thread -> (row, 4 columns), row-major, so the partial reads and the
  // output stores are coalesced and the ksplit loads of a thread are independent
  const int et = threadIdx.x - 64;
  const int rows_live = min(BM, g.M - m0);
  const float* p0 = g.ws + (long long)tile * g.ksplit * BM * BN;
  constexpr long long sstride = (long long)BM * BN;
  if (!g.gated) {
    constexpr int UPR = BN / 4;
    for (int u = et; u < rows_live * UPR; u += kEpiThreads) {
      const int r = u / UPR, c = (u % UPR) * 4;
      if (n0 + c >= g.N) continue;
      float v[4];
      sum_splits4(v, p0 + r * BN + c, sstride, g.ksplit);
      if (g.bias != nullptr) add_bias4(v, g.bias, g.bias_dtype, n0 + c, g.N);
      if (g.act != FO1_EPI_NONE) {
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = apply_act(v[j], g.act);
      }
      store_row4(g, v, m0 + r, n0 + c, g.N);
    }
  } else if constexpr (BN >= 64) {
    // gate and up columns of a 64-column pair: out[:, (n0 + c) / 2 + j] = act(gate_j) * up_j
    constexpr int UPR = BN / 8;
    for (int u = et; u < rows_live * UPR; u += kEpiThreads) {
      const int r = u / UPR, q = u % UPR;
      const int c = (q >> 3) * 64 + (q & 7) * 4;   // gate column inside the tile; up = +32
      if (n0 + c >= g.N) continue;
      float gt[4], v[4];
      sum_splits4(gt, p0 + r * BN + c, sstride, g.ksplit);
      sum_splits4(v, p0 + r * BN + c + 32, sstride, g.ksplit);
      if (g.bias != nullptr) {
        add_bias4(gt, g.bias, g.bias_dtype, n0 + c, g.N);
        add_bias4(v, g.bias, g.bias_dtype, n0 + c + 32, g.N);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = apply_act(gt[j], g.act) * v[j];
      store_row4(g, v, m0 + r, ((n0 + (c & ~63)) >> 1) + (c & 31), g.N >> 1);
    }
  }
}

// one epilogue warp's share of a finished 128 x BN accumulator (TMEM lanes of its quarter, its half of the columns): bias, activation /
// gate, residual, bf16 or fp32 stores (rows staged through shared memory into full 128-byte lines when `coalesce`)
template <int BN>
__device__ __forceinline__ void epilogue_tile(const GemmArgs& g, uint8_t* staging, int warp, int lane, uint32_t taddr, int m0, int n0) {
  const int quarter = warp & 3;
  const int half = (warp - 2) >> 2;
  constexpr bool kSplit32 = BN >= 64, kSplit64 = BN >= 128;
  const int p_beg = kSplit32 ? half * (BN / 2) : 0, p_end = kSplit32 ? (half + 1) * (BN / 2) : (half == 0 ? BN : 0);
  const int g_cut = (BN == 192) ? 128 : BN / 2;
  const int g_beg = kSplit64 ? half * g_cut : 0, g_end = kSplit64 ? (half == 0 ? g_cut : BN) : (half == 0 ? BN : 0);
  const int m = m0 + quarter * 32 + lane;
  if (!g.gated) {
    // software pipeline: the TMEM load of chunk c+1 is in flight while chunk c is converted and stored
    constexpr int NCH = (kSplit32 ? BN / 2 : BN) / 32;
    uint8_t* stg = staging + (warp - 2) * 4096;
    uint32_t r[2][32];
    const int cbeg = p_beg;
    const bool worker = p_end > p_beg;
    if (worker && n0 + cbeg < g.N) ptx::tmem_ld_32x32(taddr + cbeg, r[0]);
#pragma unroll
    for (int ci = 0; ci < NCH; ++ci) {
      const int c = cbeg + ci * 32;
      if (!worker || n0 + c >= g.N) break;  // warp-uniform
      ptx::tmem_ld_wait();
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[ci & 1][j]);
      if (ci + 1 < NCH && n0 + c + 32 < g.N) ptx::tmem_ld_32x32(taddr + c + 32, r[(ci + 1) & 1]);
      if (g.bias != nullptr) add_bias32(v, g.bias, g.bias_dtype, n0 + c, g.N);
      apply_act32(v, g.act);
      if (!g.coalesce) {
        if (m < g.M) store_row32(g, v, m, n0 + c, g.N);
      } else if (g.d_dtype == FO1_BF16) {
        // two 32-column chunks (2 x 64 B) fill a 128-byte row before it is flushed
        stage_row32(stg, lane, (ci & 1) * 4, v, true);
        const bool last = (ci + 1 == NCH) || (n0 + c + 32 >= g.N);
        if ((ci & 1) || last) flush_rows(g, stg, lane, (ci & 1) ? 8 : 4, m0 + quarter * 32, n0 + c - (ci & 1) * 32, g.N);
      } else {
        stage_row32(stg, lane, 0, v, false);
        flush_rows(g, stg, lane, 8, m0 + quarter * 32, n0 + c, g.N);
      }
    }
  } else {
    // W rows interleave [32 gate | 32 up] blocks: out[:, (n0+c)/2 + j] = act(gate_j) * up_j
#pragma unroll 1
    for (int c = g_beg; c < g_end; c += 64) {
      if (n0 + c >= g.N) break;
      uint32_t rg[32], ru[32];
      ptx::tmem_ld_32x32(taddr + c, rg);
      ptx::tmem_ld_32x32(taddr + c + 32, ru);
      ptx::tmem_ld_wait();
      float gt[32], v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) { gt[j] = __uint_as_float(rg[j]); v[j] = __uint_as_float(ru[j]); }
      if (g.bias != nullptr) {
        add_bias32(gt, g.bias, g.bias_dtype, n0 + c, g.N);
        add_bias32(v, g.bias, g.bias_dtype, n0 + c + 32, g.N);
      }
      apply_act32(gt, g.act);
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = gt[j] * v[j];
      if (!g.coalesce) {
        if (m < g.M) store_row32(g, v, m, (n0 + c) >> 1, g.N >> 1);
      } else {
        uint8_t* stg = staging + (warp - 2) * 4096;
        const bool bf = g.d_dtype == FO1_BF16;
        stage_row32(stg, lane, 0, v, bf);
        flush_rows(g, stg, lane, bf ? 4 : 8, m0 + quarter * 32, (n0 + c) >> 1, g.N >> 1);
      }
    }
  }
}

// one A tile into a ring stage: rows m0 .. m0+127 of the [M][K] matrix, or (implicit conv) the shifted pixel patch of the k-block's tap
__device__ __forceinline__ void load_a_tile(const GemmArgs& g, const CUtensorMap* tmA, uint32_t dst, uint32_t bar, int kb, int m0) {
  if (g.conv_cpb == 0) {
    ptx::tma_load_2d(dst, tmA, bar, kb * BK, m0);
  } else {
    const int tap = kb / g.conv_cpb, c0 = (kb - tap * g.conv_cpb) * BK;
    const int hw = g.conv_H * g.conv_W;
    const int b = m0 / hw, rem = m0 - b * hw;
    const int y0 = rem / g.conv_W, x0 = rem - y0 * g.conv_W;
    ptx::tma_load_4d(dst, tmA, bar, c0, x0 + tap % 3 - 1, y0 + tap / 3 - 1, b);
  }
}

template <int BN>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ GemmArgs g) {
  using Cfg = GemmCfg<BN>;
  const int S = g.stages;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: required by the 128B swizzle atoms the UMMA descriptors assume
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + S * g.a_stage_bytes;
  uint8_t* tail = smem + S * (g.a_stage_bytes + g.b_stage_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);
  uint64_t* full_bar = bars;                          // [S]
  uint64_t* empty_bar = bars + kMaxStages;            // [S]
  uint64_t* tmem_full = bars + 2 * kMaxStages;        // [2]
  uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;   // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
  volatile int* last_flag = reinterpret_cast<volatile int*>(tmem_ptr + 1);
  uint8_t* staging = tail + 512;   // [8 epilogue warps][32 rows][128 B]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int num_tiles = g.tiles_m * g.tiles_n * g.ksplit;   // work items
  const int num_kb_total = (g.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(ptx::smem_u32(full_bar + s), 1);
      ptx::mbar_init(ptx::smem_u32(empty_bar + s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(ptx::smem_u32(tmem_full + a), 1);
      ptx::mbar_init(ptx::smem_u32(tmem_empty + a), kEpiThreads / 32);  // one arrive per epilogue warp
    }
    ptx::mbar_fence_init();
  }
  if (warp == 1) ptx::tmem_alloc(ptx::smem_u32(tmem_ptr), Cfg::kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  griddep_launch();   // programmatic dependent launch: the next kernel of the stream may begin its own prologue now

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (ptx::elect_one()) {
      uint32_t it = 0;
      bool first = true;
      for (int work = blockIdx.x; work < num_tiles; work += gridDim.x) {
        const int tile = work / g.ksplit, split = work - tile * g.ksplit;
        const int m0 = (tile / g.tiles_n) * BM;
        const int n0 = (tile % g.tiles_n) * BN;
        const int kb0 = split * g.kb_per_split, kb1 = min(num_kb_total, kb0 + g.kb_per_split);
        int kb = kb0;
        if (first) {
          // W never depends on the previous kernel of the stream: fill the ring with weight tiles BEFORE waiting for
          // it to finish, then add the A tiles to the same barriers (all slots are free on the first lap)
          first = false;
          const int pre = min(S, kb1 - kb0);
          for (int i = 0; i < pre; ++i) {
            const uint32_t fb = ptx::smem_u32(full_bar + i);
            ptx::mbar_expect_tx(fb, (uint32_t)g.stage_tx);
            ptx::tma_load_2d(ptx::smem_u32(smem_b + i * g.b_stage_bytes), &tmW, fb, (kb0 + i) * BK, n0);
          }
          griddep_wait();
          for (int i = 0; i < pre; ++i)
            load_a_tile(g, &tmA, ptx::smem_u32(smem_a + i * g.a_stage_bytes), ptx::smem_u32(full_bar + i), kb0 + i, m0);
          it = pre; kb = kb0 + pre;
        }
        for (; kb < kb1; ++kb, ++it) {
          const uint32_t s = it % S, ph = (it / S) & 1;
          ptx::mbar_wait(ptx::smem_u32(empty_bar + s), ph ^ 1);
          const uint32_t fb = ptx::smem_u32(full_bar + s);
          ptx::mbar_expect_tx(fb, (uint32_t)g.stage_tx);
          load_a_tile(g, &tmA, ptx::smem_u32(smem_a + s * g.a_stage_bytes), fb, kb, m0);
          ptx::tma_load_2d(ptx::smem_u32(smem_b + s * g.b_stage_bytes), &tmW, fb, kb * BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer ======================================
    constexpr uint32_t idesc = ptx::umma_idesc_bf16(BM, BN);
    uint32_t it = 0, tcount = 0;
    for (int work = blockIdx.x; work < num_tiles; work += gridDim.x, ++tcount) {
      const int split = work % g.ksplit;
      const int kb0 = split * g.kb_per_split, kb1 = min(num_kb_total, kb0 + g.kb_per_split);
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      ptx::mbar_wait(ptx::smem_u32(tmem_empty + acc), aph ^ 1);  // epilogue has drained this accumulator
      ptx::tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * BN;
      for (int kb = kb0; kb < kb1; ++kb, ++it) {
        const uint32_t s = it % S, ph = (it / S) & 1;
        ptx::mbar_wait(ptx::smem_u32(full_bar + s), ph);
        ptx::tc_fence_after();
        if (ptx::elect_one()) {
          const uint32_t a_addr = ptx::smem_u32(smem_a + s * g.a_stage_bytes);
          const uint32_t b_addr = ptx::smem_u32(smem_b + s * g.b_stage_bytes);
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t da = ptx::umma_desc_k_sw128(a_addr + k * UMMA_K * 2);
            const uint64_t db = ptx::umma_desc_k_sw128(b_addr + k * UMMA_K * 2);
            ptx::tc_mma_bf16(tmem_d, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          ptx::tc_commit(ptx::smem_u32(empty_bar + s));                    // slot free when these MMAs retire
          if (kb == kb1 - 1) ptx::tc_commit(ptx::smem_u32(tmem_full + acc));  // accumulator complete
        }
        __syncwarp();
      }
    }
  } else {
    // ======================================= epilogue ========================================
    const int quarter = warp & 3;          // TMEM lane quarter this warp may read (hardware rule: warp id mod 4)
    const int half = (warp - 2) >> 2;      // two warps share a quarter: each owns one half of the tile's columns
    // column range of this warp: plain / split-K work in 32-column units, the gated epilogue in 64-column pairs;
    // tiles too narrow to split leave the second warp of a quarter idle (it still takes part in the barriers)
    constexpr bool kSplit32 = BN >= 64, kSplit64 = BN >= 128;
    const int p_beg = kSplit32 ? half * (BN / 2) : 0, p_end = kSplit32 ? (half + 1) * (BN / 2) : (half == 0 ? BN : 0);
    // (BN = 192: the gated split must fall on a 64-column pair boundary -> 128 + 64)
    const int g_cut = (BN == 192) ? 128 : BN / 2;
    const int g_beg = kSplit64 ? half * g_cut : 0, g_end = kSplit64 ? (half == 0 ? g_cut : BN) : (half == 0 ? BN : 0);
    uint32_t tcount = 0;
    griddep_wait();   // residual reads / output writes are ordered after the previous kernel
    for (int work = blockIdx.x; work < num_tiles; work += gridDim.x, ++tcount) {
      const int tile = work / g.ksplit, split = work - tile * g.ksplit;
      const int m0 = (tile / g.tiles_n) * BM;
      const int n0 = (tile % g.tiles_n) * BN;
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      ptx::mbar_wait(ptx::smem_u32(tmem_full + acc), aph);
      ptx::tc_fence_after();
      const int m = m0 + quarter * 32 + lane;
      const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(quarter * 32) << 16);
      if (g.ksplit > 1) {
        // ---- split-K: park the fp32 partial, the last split to arrive reduces + finishes the tile ----
        float* part = g.ws + ((long long)(tile * g.ksplit + split) * BM + quarter * 32 + lane) * BN;
#pragma unroll 1
        for (int c = p_beg; c < p_end; c += 32) {
          uint32_t r[32];
          ptx::tmem_ld_32x32(taddr + c, r);
          ptx::tmem_ld_wait();
          if (m < g.M) {
#pragma unroll
            for (int q = 0; q < 8; ++q)
              reinterpret_cast<float4*>(part + c)[q] = make_float4(__uint_as_float(r[q * 4]), __uint_as_float(r[q * 4 + 1]),
                                                                    __uint_as_float(r[q * 4 + 2]), __uint_as_float(r[q * 4 + 3]));
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(tmem_empty + acc));   // TMEM is free again: the MMA warp moves on
        __threadfence();
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (warp == 2 && lane == 0) *last_flag = (atomicAdd(g.counters + tile, 1) == g.ksplit - 1) ? 1 : 0;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        if (*last_flag) {
          __threadfence();
          splitk_finish<BN>(g, tile, m0, n0);
          if (warp == 2 && lane == 0) g.counters[tile] = 0;   // self-cleaning for the next launch
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");   // last_flag is reused by the next work item
        continue;
      }
      epilogue_tile<BN>(g, staging, warp, lane, taddr, m0, n0);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(ptx::smem_u32(tmem_empty + acc));
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// ------------------------------------------------------------------------------------- CTA-pair variant (cta_group::2)
// Large problems: a cluster of two CTAs (one TPC) owns a 256 x 256 output tile.  Each CTA stages its own 128 rows of A and HALF of
// the weight tile (128 of its 256 rows) per k-block, the leader issues tcgen05.mma.cta_group::2 (M = 256) which reads both halves,
// and each CTA's TMEM receives its 128 accumulator rows.  A stage is 32 KB per SM instead of 48 KB for the same 524 MMA cycles:
// six stages fit where four did, so the ring covers the TMA latency the single-CTA 128 x 256 tile (92 B/clk per SM) cannot
// (DESIGN.md section 4: tensor pipe 70 % -> see profiles/README.md), and L2 -> SM operand traffic drops by a third.
//   barriers (same offsets in both CTAs): full[s] lives in the LEADER (one expect_tx of 64 KB, the four TMA loads of the pair credit
//   it); empty[s] and tmem_full[a] are signalled in BOTH CTAs by the leader's multicast commit; tmem_empty[a] lives in the leader
//   and counts the 16 epilogue warps of the pair (the peer's arrive remotely).
constexpr int kPairBN = 256, kPairStages = 6;
constexpr int kPairStageBytes = (BM * BK + (kPairBN / 2) * BK) * 2;                     // 32 KB per CTA
constexpr int kPairSmemBytes = kPairStages * kPairStageBytes + 1024 + 512 + 8 * 4096;  // + align, barriers, epilogue staging

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_bf16_tcgen05_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ GemmArgs g) {
  constexpr int BN = kPairBN, S = kPairStages;
  constexpr int kAStage = BM * BK * 2, kBStage = (BN / 2) * BK * 2;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + S * kAStage;
  uint8_t* tail = smem + S * (kAStage + kBStage);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);
  uint64_t* full_bar = bars;                          // [S]   (used in the leader)
  uint64_t* empty_bar = bars + kMaxStages;            // [S]
  uint64_t* tmem_full = bars + 2 * kMaxStages;        // [2]
  uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;   // [2]   (used in the leader)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
  uint8_t* staging = tail + 512;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = ptx::cluster_ctarank();
  const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  const int pairs_m = (g.tiles_m + 1) >> 1;
  const int num_work = pairs_m * g.tiles_n;
  const int num_kb = (g.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmW);
    for (int s = 0; s < S; ++s) {
      ptx::mbar_init(ptx::smem_u32(full_bar + s), 1);
      ptx::mbar_init(ptx::smem_u32(empty_bar + s), 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(ptx::smem_u32(tmem_full + a), 1);
      ptx::mbar_init(ptx::smem_u32(tmem_empty + a), 2 * (kEpiThreads / 32));   // the epilogue warps of BOTH CTAs
    }
    ptx::mbar_fence_init_cluster();
  }
  if (warp == 1) ptx::tmem_alloc_pair(ptx::smem_u32(tmem_ptr), 2 * BN);
  ptx::tc_fence_before();
  ptx::cluster_sync_all();       // both CTAs' barriers exist before anybody signals across the pair
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  griddep_launch();

  if (warp == 0) {
    // ===================================== TMA producer (both CTAs) =====================================
    if (ptx::elect_one()) {
      griddep_wait();
      uint32_t it = 0;
      for (int work = cluster; work < num_work; work += n_clusters) {
        const int m0 = (work / g.tiles_n) * (2 * BM) + (int)rank * BM;
        const int n0 = (work % g.tiles_n) * BN + (int)rank * (BN / 2);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t s = it % S, ph = (it / S) & 1;
          ptx::mbar_wait(ptx::smem_u32(empty_bar + s), ph ^ 1);
          const uint32_t fb_local = ptx::smem_u32(full_bar + s);
          if (rank == 0) ptx::mbar_expect_tx(fb_local, 2u * (uint32_t)(kAStage + kBStage));
          const uint32_t fb = ptx::mapa_rank(fb_local, 0);
          const uint32_t dst_a = ptx::smem_u32(smem_a + s * kAStage);
          if (g.conv_cpb == 0) {
            ptx::tma_load_2d_pair(dst_a, &tmA, fb, kb * BK, m0);
          } else {
            const int tap = kb / g.conv_cpb, c0 = (kb - tap * g.conv_cpb) * BK;
            const int hw = g.conv_H * g.conv_W;
            const int b = m0 / hw, rem = m0 - b * hw;
            const int y0 = rem / g.conv_W, x0 = rem - y0 * g.conv_W;
            ptx::tma_load_4d_pair(dst_a, &tmA, fb, c0, x0 + tap % 3 - 1, y0 + tap / 3 - 1, b);
          }
          ptx::tma_load_2d_pair(ptx::smem_u32(smem_b + s * kBStage), &tmW, fb, kb * BK, n0);
        }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer (leader only) ======================================
    if (rank == 0) {
      constexpr uint32_t idesc = ptx::umma_idesc_bf16(2 * BM, BN);
      uint32_t it = 0, tcount = 0;
      for (int work = cluster; work < num_work; work += n_clusters, ++tcount) {
        const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
        ptx::mbar_wait(ptx::smem_u32(tmem_empty + acc), aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
          const uint32_t s = it % S, ph = (it / S) & 1;
          ptx::mbar_wait(ptx::smem_u32(full_bar + s), ph);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t a_addr = ptx::smem_u32(smem_a + s * kAStage);
            const uint32_t b_addr = ptx::smem_u32(smem_b + s * kBStage);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t da = ptx::umma_desc_k_sw128(a_addr + k * UMMA_K * 2);
              const uint64_t db = ptx::umma_desc_k_sw128(b_addr + k * UMMA_K * 2);
              ptx::tc_mma_bf16_pair(tmem_d, da, db, idesc, (kb > 0 || k > 0) ? 1u : 0u);
            }
            ptx::tc_commit_pair(ptx::smem_u32(empty_bar + s), 3);                      // both CTAs may refill the slot
            if (kb == num_kb - 1) ptx::tc_commit_pair(ptx::smem_u32(tmem_full + acc), 3);  // both CTAs' accumulator halves are complete
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ======================================= epilogue (both CTAs) ========================================
    const int quarter = warp & 3;
    uint32_t tcount = 0;
    griddep_wait();
    for (int work = cluster; work < num_work; work += n_clusters, ++tcount) {
      const int m0 = (work / g.tiles_n) * (2 * BM) + (int)rank * BM;
      const int n0 = (work % g.tiles_n) * BN;
      const uint32_t acc = tcount & 1, aph = (tcount >> 1) & 1;
      ptx::mbar_wait(ptx::smem_u32(tmem_full + acc), aph);
      ptx::tc_fence_after();
      const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(quarter * 32) << 16);
      if (m0 < g.M) epilogue_tile<BN>(g, staging, warp, lane, taddr, m0, n0);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(ptx::mapa_rank(ptx::smem_u32(tmem_empty + acc), 0));
    }
  }

  ptx::tc_fence_before();
  ptx::cluster_sync_all();       // the peer's MMAs read this CTA's shared memory and TMEM until the very end
  if (warp == 1) ptx::tmem_dealloc_pair(tmem_base, 2 * BN);
}

// ---------------------------------------------------------------------------------------------- host
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_tmapEncodeTiled get_encode_fn() {
  static PFN_tmapEncodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  return fn;
}

// 2-D bf16 tensor map over a row-major [outer][inner] matrix with row pitch ld (elements), 128B swizzle.
int make_tmap_2d_bf16(CUtensorMap* out, const void* ptr, uint64_t inner, uint64_t outer, uint64_t ld,
                      uint32_t box_inner, uint32_t box_outer) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return FO1_ERR_CUDA;
  }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): ptr=%p inner=%llu outer=%llu ld=%llu box=%ux%u", (int)r, ptr,
              (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)ld, box_inner, box_outer);
    return FO1_ERR_CUDA;
  }
  return FO1_OK;
}

// 3-D bf16 tensor map (attention operands: (head_dim, head, row)), 128B swizzle; out-of-range elements read as zero.
int make_tmap_3d_bf16(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                      uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return FO1_ERR_CUDA;
  }
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(3d) failed (%d): ptr=%p dims=%llu,%llu,%llu strides=%llu,%llu box=%u,%u,%u", (int)r, ptr,
              (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, (unsigned long long)stride1_bytes,
              (unsigned long long)stride2_bytes, b0, b1, b2);
    return FO1_ERR_CUDA;
  }
  return FO1_OK;
}

// 4-D bf16 tensor map over an NHWC map (channel, x, y, image), 128B swizzle; out-of-range coordinates (the conv padding) read as zero.
int make_tmap_4d_bf16(CUtensorMap* out, const void* ptr, uint64_t C, uint64_t W, uint64_t H, uint64_t B, uint32_t bc, uint32_t bw, uint32_t bh) {
  PFN_tmapEncodeTiled fn = get_encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return FO1_ERR_CUDA;
  }
  cuuint64_t dims[4] = {C, W, H, B};
  cuuint64_t strides[3] = {C * 2, W * C * 2, H * W * C * 2};
  cuuint32_t box[4] = {bc, bw, bh, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(4d) failed (%d): ptr=%p dims=%llu,%llu,%llu,%llu box=%u,%u,%u", (int)r, ptr, (unsigned long long)C,
              (unsigned long long)W, (unsigned long long)H, (unsigned long long)B, bc, bw, bh);
    return FO1_ERR_CUDA;
  }
  return FO1_OK;
}

int device_sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      sms = 148;
  }
  return sms;
}

// split-K scratch: fp32 partials + per-tile arrival counters, one set per stream (GEMMs on one stream are ordered)
struct SplitKScratch { float* ws = nullptr; size_t bytes = 0; int* counters = nullptr; };
static int splitk_scratch(cudaStream_t stream, size_t need_bytes, int need_counters, SplitKScratch** out) {
  static std::map<cudaStream_t, SplitKScratch> pool;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  SplitKScratch& sc = pool[stream];
  constexpr int kCounters = 1 << 16;
  if (need_counters > kCounters) { set_error("split-K: too many tiles (%d)", need_counters); return FO1_ERR_UNSUPPORTED; }
  if (sc.counters == nullptr) {
    FO1_CUDA(cudaMalloc(reinterpret_cast<void**>(&sc.counters), kCounters * sizeof(int)));
    FO1_CUDA(cudaMemset(sc.counters, 0, kCounters * sizeof(int)));
  }
  if (need_bytes > sc.bytes) {
    FO1_CUDA(cudaStreamSynchronize(stream));
    if (sc.ws) FO1_CUDA(cudaFree(sc.ws));
    sc.ws = nullptr; sc.bytes = 0;
    const size_t want = std::max(need_bytes, (size_t)32 << 20);
    FO1_CUDA(cudaMalloc(reinterpret_cast<void**>(&sc.ws), want));
    sc.bytes = want;
  }
  *out = &sc;
  return FO1_OK;
}

struct ConvInfo { int B, H, W, C, Wt; };   // implicit 3x3 conv: d->A is the NHWC map, d->M = B*H*W, d->K = 9*C

// the GemmArgs fields both kernels take from the descriptor and the conv geometry; tiling, ring stages and split-K are
// left zero for the launcher to plan
static GemmArgs gemm_args(const fo1_gemm_desc* d, const ConvInfo* conv) {
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.M = d->M; g.N = d->N; g.K = d->K;
  g.D = d->D; g.ldd = d->ldd; g.d_dtype = d->d_dtype;
  g.bias = d->bias; g.bias_dtype = d->bias_dtype;
  g.act = d->act;
  g.residual = static_cast<const __nv_bfloat16*>(d->residual); g.ldr = d->ldr;
  g.gated = d->gated;
  g.conv_cpb = conv ? conv->C / BK : 0; g.conv_H = conv ? conv->H : 0; g.conv_W = conv ? conv->W : 0; g.conv_Wt = conv ? conv->Wt : 0;
  g.tiles_m = ceil_div(d->M, BM);
  const int esz = d->d_dtype == FO1_BF16 ? 2 : 4;
  const bool d_ok = (reinterpret_cast<uintptr_t>(d->D) & 15) == 0 && (d->ldd * esz) % 16 == 0;
  const bool r_ok = d->residual == nullptr || ((reinterpret_cast<uintptr_t>(d->residual) & 15) == 0 && (d->ldr * 2) % 16 == 0);
  g.coalesce = (d_ok && r_ok) ? 1 : 0;
  return g;
}

template <int BN>
static int launch_gemm(const fo1_gemm_desc* d, cudaStream_t stream, int ksplit = 1, const ConvInfo* conv = nullptr) {
  using Cfg = GemmCfg<BN>;
  static bool attr_set = false;
  if (!attr_set) {
    FO1_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    attr_set = true;
  }
  CUtensorMap tmA, tmW;
  // one m-tile only (decode: M = batch): fetch just the live rows of A, rounded to the 8-row swizzle atom; the UMMA
  // still multiplies all 128 smem rows, rows >= M hold stale data whose results are never stored
  const int a_rows = d->M < BM ? ((d->M + 7) & ~7) : BM;
  if (conv != nullptr) {
    FO1_TRY(make_tmap_4d_bf16(&tmA, d->A, (uint64_t)conv->C, (uint64_t)conv->W, (uint64_t)conv->H, (uint64_t)conv->B, BK, (uint32_t)conv->Wt, (uint32_t)(BM / conv->Wt)));
  } else {
    FO1_TRY(make_tmap_2d_bf16(&tmA, d->A, (uint64_t)d->K, (uint64_t)d->M, (uint64_t)d->lda, BK, a_rows));
  }
  FO1_TRY(make_tmap_2d_bf16(&tmW, d->W, (uint64_t)d->K, (uint64_t)d->N, (uint64_t)d->ldw, BK, BN));
  GemmArgs g = gemm_args(d, conv);
  g.tiles_n = ceil_div(d->N, BN);
  g.stage_tx = (a_rows + BN) * BK * 2;
  // the UMMA reads all 128 A rows of a stage: keep the full 16 KB slot unless only the live rows are loaded AND the
  // rows beyond them may alias the next stage's data (harmless: those accumulator rows are never stored)
  g.a_stage_bytes = (a_rows < BM) ? ((a_rows * BK * 2 + 1023) & ~1023) : BM * BK * 2;
  g.b_stage_bytes = BN * BK * 2;
  {
    const int budget = Cfg::kSmemBytes - 1024 - 512 - Cfg::kStagingBytes;
    int st = budget / (g.a_stage_bytes + g.b_stage_bytes);
    // the last stage's A slot is read 16 KB deep by the UMMA: keep that window inside the operand area
    while (st > 2 && st * (g.a_stage_bytes + g.b_stage_bytes) + (BM * BK * 2 - g.a_stage_bytes) > budget) --st;
    g.stages = st < kMaxStages ? st : kMaxStages;
  }
  const int num_kb = ceil_div(d->K, BK);
  g.kb_per_split = ceil_div(num_kb, ksplit);
  g.ksplit = ceil_div(num_kb, g.kb_per_split);   // every split owns at least one k-block
  if (g.ksplit > 1) {
    SplitKScratch* sc = nullptr;
    FO1_TRY(splitk_scratch(stream, (size_t)g.tiles_m * g.tiles_n * g.ksplit * BM * BN * sizeof(float), g.tiles_m * g.tiles_n, &sc));
    g.ws = sc->ws; g.counters = sc->counters;
  }
  const int tiles = g.tiles_m * g.tiles_n * g.ksplit;
  const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
  char tag[96] = "gemm";
  if (g_prof_on) snprintf(tag, sizeof(tag), "%s:%dx%dx%d%s%s", d->M <= 128 ? "gemm_skinny" : "gemm", d->M, d->N, d->K, d->gated ? ":gated" : "", conv ? ":conv3x3" : "");
  ProfScope prof(tag, 2.0 * d->M * (double)d->N * d->K,
                 2.0 * ((double)d->M * d->K + (double)d->N * d->K + (double)d->M * (d->gated ? d->N / 2 : d->N)), stream);
  launch_k(gemm_bf16_tcgen05_kernel<BN>, dim3(grid), dim3(kGemmThreads), Cfg::kSmemBytes, stream, tmA, tmW, g);
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}

// the CTA-pair kernel: ordinary (and implicit-conv) problems with >= one wave of 256 x 256 tile pairs
static int launch_gemm_pair(const fo1_gemm_desc* d, cudaStream_t stream, const ConvInfo* conv) {
  static bool attr_set = false;
  if (!attr_set) {
    FO1_CUDA(cudaFuncSetAttribute(gemm_bf16_tcgen05_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPairSmemBytes));
    attr_set = true;
  }
  CUtensorMap tmA, tmW;
  if (conv != nullptr) {
    FO1_TRY(make_tmap_4d_bf16(&tmA, d->A, (uint64_t)conv->C, (uint64_t)conv->W, (uint64_t)conv->H, (uint64_t)conv->B, BK, (uint32_t)conv->Wt, (uint32_t)(BM / conv->Wt)));
  } else {
    FO1_TRY(make_tmap_2d_bf16(&tmA, d->A, (uint64_t)d->K, (uint64_t)d->M, (uint64_t)d->lda, BK, BM));
  }
  FO1_TRY(make_tmap_2d_bf16(&tmW, d->W, (uint64_t)d->K, (uint64_t)d->N, (uint64_t)d->ldw, BK, kPairBN / 2));
  GemmArgs g = gemm_args(d, conv);
  g.tiles_n = ceil_div(d->N, kPairBN);
  g.ksplit = 1; g.kb_per_split = ceil_div(d->K, BK);
  g.stages = kPairStages;
  const int work = ((g.tiles_m + 1) / 2) * g.tiles_n;
  const int clusters = std::min(work, device_sm_count() / 2);
  char tag[96] = "gemm";
  if (g_prof_on) snprintf(tag, sizeof(tag), "gemm:%dx%dx%d%s%s:pair", d->M, d->N, d->K, d->gated ? ":gated" : "", conv ? ":conv3x3" : "");
  ProfScope prof(tag, 2.0 * d->M * (double)d->N * d->K,
                 2.0 * ((double)d->M * d->K + (double)d->N * d->K + (double)d->M * (d->gated ? d->N / 2 : d->N)), stream);
  launch_k(gemm_bf16_tcgen05_pair_kernel, dim3(2 * clusters), dim3(kGemmThreads), kPairSmemBytes, stream, tmA, tmW, g);
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}
// one wave of tile pairs at least, and whole 128-row A boxes
static bool use_pair_kernel(int M, int N) {
  const long long work = (long long)ceil_div(ceil_div(M, BM), 2) * ceil_div(N, kPairBN);
  return M >= BM && N >= kPairBN && work >= device_sm_count() / 2;
}

int gemm_bf16(const fo1_gemm_desc* d, cudaStream_t stream) {
  FO1_CHECK_ARG(d != nullptr, "fo1_gemm_bf16: null descriptor");
  FO1_CHECK_ARG(d->M >= 0 && d->N > 0 && d->K > 0, "fo1_gemm_bf16: bad shape M=%d N=%d K=%d", d->M, d->N, d->K);
  if (d->M == 0) return FO1_OK;
  FO1_CHECK_ARG(d->A && d->W && d->D, "fo1_gemm_bf16: null operand");
  FO1_CHECK_ARG((reinterpret_cast<uintptr_t>(d->A) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->W) & 15) == 0,
                "fo1_gemm_bf16: A and W must be 16-byte aligned");
  FO1_CHECK_ARG(d->lda >= d->K && d->ldw >= d->K && (d->lda % 8) == 0 && (d->ldw % 8) == 0,
                "fo1_gemm_bf16: lda=%lld / ldw=%lld must be >= K and multiples of 8 elements (TMA 16-byte pitch)",
                (long long)d->lda, (long long)d->ldw);
  FO1_CHECK_ARG(d->d_dtype == FO1_BF16 || d->d_dtype == FO1_F32, "fo1_gemm_bf16: d_dtype %d unsupported", d->d_dtype);
  FO1_CHECK_ARG(d->bias == nullptr || d->bias_dtype == FO1_BF16 || d->bias_dtype == FO1_F32, "fo1_gemm_bf16: bias_dtype %d unsupported", d->bias_dtype);
  FO1_CHECK_ARG(d->act >= FO1_EPI_NONE && d->act <= FO1_EPI_SILU, "fo1_gemm_bf16: act %d unsupported", d->act);
  const int n_out = d->gated ? d->N / 2 : d->N;
  FO1_CHECK_ARG(!d->gated || d->N % 64 == 0, "fo1_gemm_bf16: gated N=%d must be a multiple of 64", d->N);
  FO1_CHECK_ARG(d->ldd >= n_out, "fo1_gemm_bf16: ldd=%lld < %d", (long long)d->ldd, n_out);
  FO1_CHECK_ARG(d->residual == nullptr || d->ldr >= n_out, "fo1_gemm_bf16: ldr too small");
  if (d->tile_n != 0) {   // pinned by the caller (tuning sweeps, tests of the split-K / tile variants)
    const int ks = d->split_k > 0 ? d->split_k : 1;
    FO1_CHECK_ARG(!d->gated || d->tile_n >= 64, "fo1_gemm_bf16: gated needs tile_n >= 64");
    FO1_CHECK_ARG(ks == 1 || (long long)ceil_div(d->M, BM) * ceil_div(d->N, d->tile_n) <= (1 << 16), "fo1_gemm_bf16: too many tiles for split_k");
    switch (d->tile_n) {
      case 32: return launch_gemm<32>(d, stream, ks);
      case 64: return launch_gemm<64>(d, stream, ks);
      case 128: return launch_gemm<128>(d, stream, ks);
      case 192: return launch_gemm<192>(d, stream, ks);
      case 256: return launch_gemm<256>(d, stream, ks);
      default: set_error("fo1_gemm_bf16: tile_n=%d unsupported (32, 64, 128, 192, 256)", d->tile_n); return FO1_ERR_INVALID_ARG;
    }
  }
  // tile-width choice: widest tile that still yields >= 1 wave of CTAs, else narrower for occupancy
  const int sms = device_sm_count();
  const long long tm = ceil_div(d->M, BM);
  if (use_pair_kernel(d->M, d->N)) return launch_gemm_pair(d, stream, nullptr);
  if (d->N >= 256 && tm * ceil_div(d->N, 256) >= sms) return launch_gemm<256>(d, stream);
  // weight-streaming problems whose 128-wide tiles need a second, mostly empty wave (decode gate/up: 172 tiles on 148 SMs)
  // run as ONE wave of 192-wide tiles instead (measured 27.3 -> 22.3 us, profiles/r01_sweep_skinny.json)
  if (tm == 1 && d->N >= 192 && ceil_div(d->N, 128) > sms && ceil_div(d->N, 192) <= sms) return launch_gemm<192>(d, stream);
  if (d->N >= 128 && tm * ceil_div(d->N, 128) >= sms) return launch_gemm<128>(d, stream);
  if (d->gated || tm * ceil_div(d->N, 64) >= sms) return launch_gemm<64>(d, stream);
  // skinny problems (decode: M = batch, weight streaming): 64-wide tiles (the activation tile every CTA re-reads is
  // half the weight tile) and split-K until one wave of CTAs pulls weights, >= 8 k-blocks per split so the ring
  // still fills (measured: scripts/sweep_skinny.py, profiles/r01_sweep_skinny.json)
  const int bn = d->N >= 512 ? 64 : 32;
  const long long t = tm * ceil_div(d->N, bn);
  int ks = 1;
  // (only inside a SplitKScope -- decode steps, LM head, the public entry point: see common.cuh)
  if (t_splitk_ok && t * 2 <= sms) ks = (int)std::min<long long>(std::min<long long>(8, sms / t), std::max(1, ceil_div(d->K, BK) / 8));
  return bn == 64 ? launch_gemm<64>(d, stream, ks) : launch_gemm<32>(d, stream, ks);
}

// out[(b, y, x)][n] = sum_{ky, kx, c} x[b][y + ky - 1][x + kx - 1][c] * W[n][(ky * 3 + kx) * C + c]   (3x3, pad 1, stride 1, NHWC, no bias)
// as an implicit GEMM: no column matrix, the A tiles are shifted patches of the map (zero padding = the TMA's out-of-range fill).
// Returns FO1_ERR_UNSUPPORTED-like -1000 when the shape does not tile (caller falls back to im2col + linear).
int conv3x3_gemm(const bf16* x, int B, int H, int W, int C, const bf16* Wm, bf16* out, long long ldo, int N, cudaStream_t stream) {
  const bool fits = C % BK == 0 && (H * W) % BM == 0 && ((W % BM == 0) || (BM % W == 0 && H % (BM / W) == 0)) && N % 8 == 0;
  if (!fits) return -1000;
  if ((long long)B * H * W == 0) return FO1_OK;
  FO1_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(Wm) & 15) == 0, "conv3x3_gemm: operands must be 16-byte aligned");
  fo1_gemm_desc d;
  memset(&d, 0, sizeof(d));
  d.M = B * H * W; d.N = N; d.K = 9 * C;
  d.A = x; d.lda = C; d.W = Wm; d.ldw = 9 * C; d.D = out; d.ldd = ldo; d.d_dtype = FO1_BF16;
  ConvInfo ci{B, H, W, C, W % BM == 0 ? BM : W};
  const int sms = device_sm_count();
  const long long tm = ceil_div(d.M, BM);
  if (use_pair_kernel(d.M, N)) return launch_gemm_pair(&d, stream, &ci);
  if (N >= 256 && tm * ceil_div(N, 256) >= sms) return launch_gemm<256>(&d, stream, 1, &ci);
  if (N >= 128 && tm * ceil_div(N, 128) >= sms) return launch_gemm<128>(&d, stream, 1, &ci);
  return launch_gemm<64>(&d, stream, 1, &ci);
}

}  // namespace fo1

extern "C" int fo1_gemm_bf16(const fo1_gemm_desc* d, void* stream) {
  fo1::SplitKScope sk(true);     // a caller's own GEMM: no batch semantics to protect
  return fo1::gemm_bf16(d, static_cast<cudaStream_t>(stream));
}

namespace fo1 {
int linear(const bf16* A, long long lda, const bf16* W, long long ldw, void* D, long long ldd, int d_dtype, int M, int N,
           int K, const void* bias, int bias_dtype, int act, const bf16* residual, long long ldr, int gated,
           cudaStream_t stream) {
  fo1_gemm_desc d;
  memset(&d, 0, sizeof(d));
  d.M = M; d.N = N; d.K = K;
  d.A = A; d.lda = lda; d.W = W; d.ldw = ldw; d.D = D; d.ldd = ldd; d.d_dtype = d_dtype;
  d.bias = bias; d.bias_dtype = bias_dtype; d.act = act; d.residual = residual; d.ldr = ldr; d.gated = gated;
  return gemm_bf16(&d, stream);
}
}  // namespace fo1
