// attention_tc.cu -- variable-length softmax attention on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// One kernel serves the ViT's windowed / full attention (head_dim 80; modeling_qwen2_5_vl.py:172-209, the
// flash_attn_varlen_func call at :205), DaViT's 12x12 window attention (head_dim 32; modeling_davit.py:225-282) and the
// LLM's causal GQA prefill (head_dim 128, 16 q / 2 kv heads; modeling_qwen2_5_vl.py:822-913, _flash_attention_forward
// at :895).
//
// Formulation: the packed token rows are cut into query tiles of up to 128 rows REGARDLESS of the segment boundaries; a
// row attends the keys [lo, hi) of its own segment (hi clipped to row + 1 when causal), so a tile's key range is
// [lo(first row), hi(last row)) and the per-row mask is two integer compares.  That makes 64-token ViT windows, ragged
// edge windows (46x46 grids), 144-token DaViT windows, whole images and ragged causal prompts the same code path.
// The engines pass a tile table whose tiling restarts at every image / prompt, so a sample's result does not depend on
// its position in the batch (bit-identical across batch compositions and rank counts).
//
// CTA = one (query tile, head), 192 threads, two CTAs per SM:
//   warp 0   : TMA producer -- Q once, then K and V 64-key tiles through two 2-stage rings (3-D tensor maps over
//              (head_dim, head, row), 64-wide boxes, 128-byte swizzle; head_dim 80 / 32 are zero-filled to the box by
//              the TMA out-of-bounds rule, so every operand has 128-byte rows);
//   warp 1   : tcgen05.mma issuer -- S_j = Q.K_j^T (M 128 x N 64, K-major operands) into one of two TMEM buffers, then
//              O += P_j.V_j with V taken MN-major straight from its TMA tile (no transposition pass) and P from shared
//              memory; tcgen05.commit publishes S / frees the ring slots / publishes O;
//   warps 2-5: softmax -- one thread per query row: tcgen05.ld of its S row, mask, running max / sum in registers,
//              P = exp2(S*scale - m) written as bf16 in the K-major swizzled layout the next MMA reads.  O stays in
//              TMEM for the whole key loop; it is rescaled (tcgen05.ld -> mul -> tcgen05.st) only when a row's max has
//              grown by more than 2^8 since the last rescale (stale maxima are exact: the factor cancels in O / l).
// Warps whose 32 rows cannot see a key tile at all (the other window of the tile) skip the exponentials.
#include <cuda.h>

#include <algorithm>
#include <map>
#include <mutex>

#include "kernels.cuh"
#include "ptx.cuh"

namespace fo1 {

int make_tmap_3d_bf16(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                      uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2);

constexpr int kAtM = 128;          // query rows per CTA
constexpr int kAtN = 64;           // keys per iteration
constexpr int kAtThreads = 192;
constexpr float kAtRescale = 8.0f; // log2 units a row maximum may lag behind before O is rescaled

template <int HD>
struct AtCfg {
  static constexpr int HDP = HD <= 64 ? 64 : 128;      // head_dim as staged (zero-filled)
  static constexpr int NDB = HDP / 64;                 // 64-wide boxes per row
  static constexpr int kQBytes = NDB * kAtM * 128;
  static constexpr int kKBytes = NDB * kAtN * 128;
  static constexpr int kVBytes = NDB * kAtN * 128;
  static constexpr int kPBytes = kAtM * 128;
  static constexpr int kTileBytes = kQBytes + 2 * kKBytes + 2 * kVBytes + kPBytes;
  // the dynamic window is at least 128-byte aligned: aligning it to 1024 costs at most 896 B; 128 B of barriers
  // follow the tiles.  head_dim 80 / 128: 115 712 B, exactly what lets two CTAs share an SM (2 x (113 KB + 1 KB)).
  static constexpr int kSmemBytes = kTileBytes + 896 + 128;
  static constexpr int kTmemCols = 256;                // S0 [0,64) | S1 [64,128) | O [128, 128 + HDP)
  static_assert(HD % 16 == 0 && HD <= 128, "head_dim must be a multiple of 16, at most 128");
};

struct AttnTcArgs {
  bf16* o; long long ldo;
  const int2* rowseg;   // [T]: keys [lo, hi) of the segment every packed row belongs to
  const int2* tiles;    // optional [n_tiles] (first row, rows <= 128) of every query tile; null: tile i = rows [128 i, 128 i + 128)
  int T, q_heads, kv_heads;
  int n_work;           // query tiles x heads
  float sl2;            // softmax scale * log2(e)
};

// a wait that turns a protocol bug into a trap instead of a hung GPU
__device__ __forceinline__ void at_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t b = ptx::smem_u32(bar);
  uint32_t spins = 0;
  while (!ptx::mbar_try_wait(b, parity)) {
    if (++spins > (1u << 26)) __trap();
  }
}

// (lo, hi) of every packed row from cu_seqlens
__global__ void __launch_bounds__(256) attn_rowseg_kernel(const int* __restrict__ cu, int n_seqs, int T, int2* __restrict__ out) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= T) return;
  int a = 0, b = n_seqs;   // largest s with cu[s] <= r
  while (b - a > 1) {
    const int mid = (a + b) >> 1;
    if (__ldg(cu + mid) <= r) a = mid; else b = mid;
  }
  const int lo = __ldg(cu + a), hi = __ldg(cu + a + 1);
  out[r] = (r >= lo && r < hi) ? make_int2(lo, hi) : make_int2(r, r + 1);   // rows outside every segment see themselves only
}

template <int HD, bool CAUSAL>
__global__ void __launch_bounds__(kAtThreads, 2)
attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
               const AttnTcArgs a) {
  using Cfg = AtCfg<HD>;
  constexpr int NDB = Cfg::NDB;
  extern __shared__ uint8_t at_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(at_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::kQBytes;
  uint8_t* sV = sK + 2 * Cfg::kKBytes;
  uint8_t* sP = sV + 2 * Cfg::kVBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + Cfg::kPBytes);
  uint64_t* q_full = bars;            // [1]
  uint64_t* k_full = bars + 1;        // [2]
  uint64_t* k_empty = bars + 3;       // [2]
  uint64_t* v_full = bars + 5;        // [2]
  uint64_t* v_empty = bars + 7;       // [2]
  uint64_t* s_full = bars + 9;        // [2]
  uint64_t* s_empty = bars + 11;      // [2]
  uint64_t* p_full = bars + 13;       // [1]
  uint64_t* o_done = bars + 14;       // [1]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(sP);   // read once before the first P tile is written (second __syncthreads below)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* q_empty = bars + 15;      // [1] the softmax warps are done with the Q tile (their output staging) and with O in TMEM

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmQ);
    ptx::prefetch_tmap(&tmK);
    ptx::prefetch_tmap(&tmV);
    ptx::mbar_init(ptx::smem_u32(q_full), 1);
    ptx::mbar_init(ptx::smem_u32(q_empty), 128);
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(ptx::smem_u32(k_full + s), 1);
      ptx::mbar_init(ptx::smem_u32(k_empty + s), 1);
      ptx::mbar_init(ptx::smem_u32(v_full + s), 1);
      ptx::mbar_init(ptx::smem_u32(v_empty + s), 1);
      ptx::mbar_init(ptx::smem_u32(s_full + s), 1);
      ptx::mbar_init(ptx::smem_u32(s_empty + s), 128);
    }
    ptx::mbar_init(ptx::smem_u32(p_full), 128);
    ptx::mbar_init(ptx::smem_u32(o_done), 1);
    ptx::mbar_fence_init();
  }
  if (warp == 1) ptx::tmem_alloc(ptx::smem_u32(tmem_ptr), Cfg::kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  __syncthreads();                    // everybody holds the TMEM address before the softmax warps reuse its slot for P

  // Persistent CTA: work items (query tile, head), head fastest, static round robin.  Barriers, TMEM and the tensor-map prefetch are
  // set up once; every role walks the same item list and carries ONE running key-tile counter g across items (ring stage = g & 1,
  // phase = (g >> 1) & 1), so the K/V ring keeps streaming across item boundaries.  Per item: the Q tile and the O accumulator are
  // single-buffered -- the producer reloads Q, and the MMA warp restarts O, only after the softmax warps released them (q_empty).
  const int n_work = a.n_work;
  auto item_geom = [&](int work, int& head, int& kvh, int& row0, int& rows_valid, int& kv_begin, int& n_kv) {
    head = work % a.q_heads;
    const int tile = work / a.q_heads;
    kvh = head / (a.q_heads / a.kv_heads);
    row0 = tile * kAtM; rows_valid = min(kAtM, a.T - row0);
    if (a.tiles != nullptr) {
      const int2 tl = __ldg(a.tiles + tile);
      row0 = tl.x; rows_valid = tl.y;
    }
    // key range of the tile (segments are ordered, so first row's lo / last row's hi bound every row's range)
    kv_begin = __ldg(&a.rowseg[row0].x);
    int kv_end = __ldg(&a.rowseg[row0 + rows_valid - 1].y);
    if (CAUSAL) kv_end = min(kv_end, row0 + rows_valid);
    n_kv = (kv_end - kv_begin + kAtN - 1) / kAtN;
  };

  if (warp == 0) {
    // ================================================ TMA producer ================================================
    if (ptx::elect_one()) {
      uint32_t g = 0, item = 0;
      for (int work = blockIdx.x; work < n_work; work += gridDim.x, ++item) {
        int head, kvh, row0, rows_valid, kv_begin, n_kv;
        item_geom(work, head, kvh, row0, rows_valid, kv_begin, n_kv);
        if (item > 0) at_wait(q_empty, (item - 1) & 1);
        ptx::mbar_expect_tx(ptx::smem_u32(q_full), Cfg::kQBytes);
#pragma unroll
        for (int b = 0; b < NDB; ++b) ptx::tma_load_3d(ptx::smem_u32(sQ + b * kAtM * 128), &tmQ, ptx::smem_u32(q_full), b * 64, head, row0);
        for (int j = 0; j < n_kv; ++j, ++g) {
          const uint32_t st = g & 1;
          const int key0 = kv_begin + j * kAtN;
          if (g >= 2) at_wait(k_empty + st, ((g >> 1) - 1) & 1);
          ptx::mbar_expect_tx(ptx::smem_u32(k_full + st), Cfg::kKBytes);
#pragma unroll
          for (int b = 0; b < NDB; ++b)
            ptx::tma_load_3d(ptx::smem_u32(sK + st * Cfg::kKBytes + b * kAtN * 128), &tmK, ptx::smem_u32(k_full + st), b * 64, kvh, key0);
          if (g >= 2) at_wait(v_empty + st, ((g >> 1) - 1) & 1);
          ptx::mbar_expect_tx(ptx::smem_u32(v_full + st), Cfg::kVBytes);
#pragma unroll
          for (int b = 0; b < NDB; ++b)
            ptx::tma_load_3d(ptx::smem_u32(sV + st * Cfg::kVBytes + b * kAtN * 128), &tmV, ptx::smem_u32(v_full + st), b * 64, kvh, key0);
        }
      }
    }
  } else if (warp == 1) {
    // ================================================= MMA issuer =================================================
    constexpr uint32_t idesc_s = ptx::umma_idesc_bf16(kAtM, kAtN);
    uint32_t gbase = 0, item = 0;
    for (int work = blockIdx.x; work < n_work; work += gridDim.x, ++item) {
      int head, kvh, row0, rows_valid, kv_begin, n_kv;
      item_geom(work, head, kvh, row0, rows_valid, kv_begin, n_kv);
      at_wait(q_full, item & 1);          // (Q is reloaded only after q_empty: O of the previous item has been read out by then)
      for (int j = 0; j <= n_kv; ++j) {
        if (j < n_kv) {                                   // S_j = Q . K_j^T
          const uint32_t g = gbase + j, st = g & 1;
          at_wait(k_full + st, (g >> 1) & 1);
          if (g >= 2) at_wait(s_empty + st, ((g >> 1) - 1) & 1);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t q_addr = ptx::smem_u32(sQ), k_addr = ptx::smem_u32(sK + st * Cfg::kKBytes);
#pragma unroll
            for (int kk = 0; kk < HD / 16; ++kk) {
              const uint64_t da = ptx::umma_desc_k_sw128(q_addr + (kk >> 2) * (kAtM * 128) + (kk & 3) * 32);
              const uint64_t db = ptx::umma_desc_k_sw128(k_addr + (kk >> 2) * (kAtN * 128) + (kk & 3) * 32);
              ptx::tc_mma_bf16(tmem_base + st * kAtN, da, db, idesc_s, kk > 0 ? 1u : 0u);
            }
            ptx::tc_commit(ptx::smem_u32(s_full + st));
            ptx::tc_commit(ptx::smem_u32(k_empty + st));
          }
          __syncwarp();
        }
        if (j >= 1) {                                     // O += P_{j-1} . V_{j-1}
          const int jj = j - 1;
          const uint32_t g = gbase + jj, st = g & 1;
          at_wait(p_full, g & 1);
          at_wait(v_full + st, (g >> 1) & 1);
          ptx::tc_fence_after();
          if (ptx::elect_one()) {
            const uint32_t p_addr = ptx::smem_u32(sP), v_addr = ptx::smem_u32(sV + st * Cfg::kVBytes);
#pragma unroll
            for (int kk = 0; kk < kAtN / 16; ++kk) {
              const uint64_t da = ptx::umma_desc_k_sw128(p_addr + kk * 32);
#pragma unroll
              for (int b = 0; b < NDB; ++b) {
                constexpr int kLastN = HD - (NDB - 1) * 64;             // live dims of the last box (16 for head_dim 80)
                const int nb = (b == NDB - 1) ? kLastN : 64;
                const uint64_t db = ptx::umma_desc_mn_sw128(v_addr + b * (kAtN * 128) + kk * 2048);
                ptx::tc_mma_bf16(tmem_base + 2 * kAtN + b * 64, da, db, ptx::umma_idesc_bf16(kAtM, nb) | ptx::kUmmaBMajorMN,
                                 (jj > 0 || kk > 0) ? 1u : 0u);
              }
            }
            ptx::tc_commit(ptx::smem_u32(o_done));
            ptx::tc_commit(ptx::smem_u32(v_empty + st));
          }
          __syncwarp();
        }
      }
      gbase += (uint32_t)n_kv;
    }
  } else {
    // ================================================== softmax ===================================================
    const int quarter = warp & 3;                       // TMEM lane quarter this warp may touch (warp id mod 4)
    const int r = quarter * 32 + lane;                  // row inside the tile == TMEM lane
    const uint32_t t_lane = tmem_base + ((uint32_t)(quarter * 32) << 16);
    uint8_t* p_row = sP + r * 128;
    uint32_t gbase = 0;
    for (int work = blockIdx.x; work < n_work; work += gridDim.x) {
      int head, kvh, row0, rows_valid, kv_begin, n_kv;
      item_geom(work, head, kvh, row0, rows_valid, kv_begin, n_kv);
      const int row = row0 + r;
      int lo = 0, hi = 0;                                 // rows beyond T: empty key range
      if (r < rows_valid) {
        const int2 rs = __ldg(a.rowseg + row);
        lo = rs.x; hi = rs.y;
        if (CAUSAL) hi = min(hi, row + 1);
      }
      int wlo_min = lo, wlo_max = lo, whi_min = hi, whi_max = hi;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wlo_min = min(wlo_min, __shfl_xor_sync(0xffffffffu, wlo_min, o));
        wlo_max = max(wlo_max, __shfl_xor_sync(0xffffffffu, wlo_max, o));
        whi_min = min(whi_min, __shfl_xor_sync(0xffffffffu, whi_min, o));
        whi_max = max(whi_max, __shfl_xor_sync(0xffffffffu, whi_max, o));
      }
      const uint32_t span = (uint32_t)(hi - lo);
      float m_run = -INFINITY, l_run = 0.f;               // running max (scaled, log2 units) and sum of this row

      for (int j = 0; j < n_kv; ++j) {
        const uint32_t g = gbase + j, st = g & 1;
        const int k0 = kv_begin + j * kAtN;
        const bool dead = (k0 >= whi_max) || (k0 + kAtN <= wlo_min);          // no row of this warp sees the tile
        const bool interior = (k0 >= wlo_max) && (k0 + kAtN <= whi_min);      // every row sees every key
        at_wait(s_full + st, (g >> 1) & 1);
        ptx::tc_fence_after();
        uint32_t sr[2][32];
        if (!dead) {
          ptx::tmem_ld_32x32(t_lane + st * kAtN, sr[0]);
          ptx::tmem_ld_32x32(t_lane + st * kAtN + 32, sr[1]);
          ptx::tmem_ld_wait();
        }
        ptx::tc_fence_before();
        ptx::mbar_arrive(ptx::smem_u32(s_empty + st));     // S_j is in registers: the buffer may take S_{j+2}
        uint32_t pk[32];
        if (dead) {
#pragma unroll
          for (int c = 0; c < 32; ++c) pk[c] = 0u;
        } else {
          float mt = -INFINITY;
          if (interior) {
#pragma unroll
            for (int c = 0; c < 64; ++c) mt = fmaxf(mt, __uint_as_float(sr[c >> 5][c & 31]));
          } else {
#pragma unroll
            for (int c = 0; c < 64; ++c) {
              const bool ok = (uint32_t)(k0 + c - lo) < span;
              const float x = ok ? __uint_as_float(sr[c >> 5][c & 31]) : -INFINITY;
              sr[c >> 5][c & 31] = __float_as_uint(x);
              mt = fmaxf(mt, x);
            }
          }
          const float m_new = fmaxf(m_run, mt * a.sl2);
          // lazy rescale: keep a stale maximum until it lags by 2^8; a row without any live key so far has O == 0 exactly
          const bool grow = m_new > m_run + kAtRescale;
          const bool touch = grow && (m_run != -INFINITY);
          float alpha = 1.0f;
          if (grow) {
            if (touch) { alpha = ex2_approx(m_run - m_new); l_run *= alpha; }
            m_run = m_new;
          }
          if (__any_sync(0xffffffffu, touch)) {            // (touch implies j >= 1: g - 1 is this item's previous tile)
            at_wait(o_done, (g - 1) & 1);                  // P_{j-1}.V_{j-1} has landed in O
            ptx::tc_fence_after();
#pragma unroll
            for (int c = 0; c < (HD + 31) / 32; ++c) {
              uint32_t orow[32];
              ptx::tmem_ld_32x32(t_lane + 2 * kAtN + c * 32, orow);
              ptx::tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) orow[i] = __float_as_uint(__uint_as_float(orow[i]) * alpha);
              ptx::tmem_st_32x32(t_lane + 2 * kAtN + c * 32, orow);
            }
            ptx::tmem_st_wait();
            ptx::tc_fence_before();
          }
          const float m_use = (m_run == -INFINITY) ? 0.f : m_run;
          float sum = 0.f;
#pragma unroll
          for (int c = 0; c < 64; c += 2) {
            const float p0 = ex2_approx(fmaf(__uint_as_float(sr[c >> 5][c & 31]), a.sl2, -m_use));
            const float p1 = ex2_approx(fmaf(__uint_as_float(sr[(c + 1) >> 5][(c + 1) & 31]), a.sl2, -m_use));
            sum += p0 + p1;
            pk[c >> 1] = pack_bf16(p0, p1);
          }
          l_run += sum;
        }
        if (g >= 1) at_wait(o_done, (g - 1) & 1);          // the previous P (of this item or the last one) has been consumed: the buffer is free
#pragma unroll
        for (int c = 0; c < 8; ++c)
          *reinterpret_cast<uint4*>(p_row + ((c ^ (r & 7)) << 4)) = make_uint4(pk[4 * c], pk[4 * c + 1], pk[4 * c + 2], pk[4 * c + 3]);
        ptx::fence_proxy_async_smem();
        ptx::mbar_arrive(ptx::smem_u32(p_full));
      }
      gbase += (uint32_t)n_kv;

      // ---- O / l -> bf16, staged through the (dead) Q tile of this warp, row-contiguous 16-byte stores ----
      at_wait(o_done, (gbase - 1) & 1);
      ptx::tc_fence_after();
      const float inv = l_run > 0.f ? 1.0f / l_run : 0.f;
      constexpr int PITCH = Cfg::HDP * 2;
      uint8_t* stg = sQ + (warp - 2) * 32 * PITCH;
#pragma unroll
      for (int c = 0; c < (HD + 31) / 32; ++c) {
        uint32_t orow[32];
        ptx::tmem_ld_32x32(t_lane + 2 * kAtN + c * 32, orow);
        ptx::tmem_ld_wait();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          if (c * 32 + q * 8 < HD) {
            const int ch = c * 4 + q;                     // 16-byte chunk of the row
            *reinterpret_cast<uint4*>(stg + lane * PITCH + (((ch & ~7) | ((ch ^ lane) & 7)) << 4)) =
                make_uint4(pack_bf16(__uint_as_float(orow[q * 8 + 0]) * inv, __uint_as_float(orow[q * 8 + 1]) * inv),
                           pack_bf16(__uint_as_float(orow[q * 8 + 2]) * inv, __uint_as_float(orow[q * 8 + 3]) * inv),
                           pack_bf16(__uint_as_float(orow[q * 8 + 4]) * inv, __uint_as_float(orow[q * 8 + 5]) * inv),
                           pack_bf16(__uint_as_float(orow[q * 8 + 6]) * inv, __uint_as_float(orow[q * 8 + 7]) * inv));
          }
        }
      }
      ptx::tc_fence_before();
      __syncwarp();
      constexpr int CH = HD / 8;
      bf16* op = a.o + (long long)(row0 + quarter * 32) * a.ldo + (long long)head * HD;
      for (int i = lane; i < 32 * CH; i += 32) {
        const int rr = i / CH, ch = i - rr * CH;
        if (quarter * 32 + rr < rows_valid)
          *reinterpret_cast<uint4*>(op + (long long)rr * a.ldo + ch * 8) =
              *reinterpret_cast<const uint4*>(stg + rr * PITCH + (((ch & ~7) | ((ch ^ rr) & 7)) << 4));
      }
      __syncwarp();
      ptx::fence_proxy_async_smem();                       // the next Q tile arrives through the async proxy
      ptx::mbar_arrive(ptx::smem_u32(q_empty));            // Q tile (staging) and O are free for the next item
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// ---------------------------------------------------------------------------------------------------------- host
// (lo, hi) table scratch: one grow-only buffer per stream (attention calls on one stream are ordered)
static int rowseg_scratch(cudaStream_t stream, size_t rows, int2** out) {
  struct Buf { int2* p = nullptr; size_t rows = 0; };
  static std::map<cudaStream_t, Buf> pool;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  Buf& b = pool[stream];
  if (rows > b.rows) {
    FO1_CUDA(cudaStreamSynchronize(stream));
    if (b.p) FO1_CUDA(cudaFree(b.p));
    b.p = nullptr; b.rows = 0;
    const size_t want = std::max<size_t>(rows, 1 << 17);
    FO1_CUDA(cudaMalloc(reinterpret_cast<void**>(&b.p), want * sizeof(int2)));
    b.rows = want;
  }
  *out = b.p;
  return FO1_OK;
}

void attention_tile_table(const std::vector<int>& group_cu, std::vector<int>& tiles) {
  tiles.clear();
  for (size_t g = 0; g + 1 < group_cu.size(); ++g)
    for (int r = group_cu[g]; r < group_cu[g + 1]; r += kAtM) {
      tiles.push_back(r);
      tiles.push_back(std::min(kAtM, group_cu[g + 1] - r));
    }
}

int attention_rowseg(const int* cu_seqlens, int n_seqs, int T, int* rowseg /*[T][2]*/, cudaStream_t s) {
  if (T <= 0) return FO1_OK;
  attn_rowseg_kernel<<<ceil_div(T, 256), 256, 0, s>>>(cu_seqlens, n_seqs, T, reinterpret_cast<int2*>(rowseg));
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}

template <int HD, bool CAUSAL>
static int launch_attn_tc(const AttnArgs& a, const int2* rowseg, cudaStream_t s) {
  using Cfg = AtCfg<HD>;
  static bool attr_set = false;
  if (!attr_set) {
    FO1_CUDA(cudaFuncSetAttribute(attn_tc_kernel<HD, CAUSAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    FO1_CUDA(cudaFuncSetAttribute(attn_tc_kernel<HD, CAUSAL>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    attr_set = true;
  }
  const int T = a.total_rows;
  CUtensorMap tmQ, tmK, tmV;
  FO1_TRY(make_tmap_3d_bf16(&tmQ, a.q, HD, a.q_heads, T, (uint64_t)HD * 2, (uint64_t)a.ldq * 2, 64, 1, kAtM));
  FO1_TRY(make_tmap_3d_bf16(&tmK, a.k, HD, a.kv_heads, T, (uint64_t)HD * 2, (uint64_t)a.ldk * 2, 64, 1, kAtN));
  FO1_TRY(make_tmap_3d_bf16(&tmV, a.v, HD, a.kv_heads, T, (uint64_t)HD * 2, (uint64_t)a.ldv * 2, 64, 1, kAtN));
  AttnTcArgs g;
  g.o = a.o; g.ldo = a.ldo; g.rowseg = rowseg; g.T = T; g.q_heads = a.q_heads; g.kv_heads = a.kv_heads;
  g.tiles = reinterpret_cast<const int2*>(a.tiles);
  g.sl2 = a.scale * 1.4426950408889634f;
  const long long blocks = (long long)(a.tiles != nullptr ? a.n_tiles : ceil_div(T, kAtM)) * a.q_heads;
  FO1_CHECK_ARG(blocks < (1ll << 31), "attention: grid too large (%lld blocks)", blocks);
  g.n_work = (int)blocks;
  ProfScope prof(CAUSAL ? "attn_causal" : "attn", a.flops, 0.0, s);
  // persistent for the non-causal shapes (equal-cost items: ViT / DaViT windows 0.40 -> 0.33 ms, 0.78 -> 0.66 ms per layer at 32 images): two
  // CTAs per SM walk the item list.  Causal prompts have items of very different cost; the static round robin lost 19 % against the
  // hardware block scheduler there, so they keep one CTA per item (the same kernel with a one-item list).
  const long long resident = 2LL * device_sm_count();
  const unsigned grid = (unsigned)((CAUSAL || blocks < resident) ? blocks : resident);
  attn_tc_kernel<HD, CAUSAL><<<grid, kAtThreads, Cfg::kSmemBytes, s>>>(tmQ, tmK, tmV, g);
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}

int attention_varlen(const AttnArgs& a, cudaStream_t s) {
  FO1_CHECK_ARG(a.q && a.k && a.v && a.o && (a.cu_seqlens || a.rowseg), "attention: null pointer");
  FO1_CHECK_ARG(a.q_heads > 0 && a.kv_heads > 0 && a.q_heads % a.kv_heads == 0, "attention: heads %d/%d", a.q_heads, a.kv_heads);
  FO1_CHECK_ARG((a.ldq % 8) == 0 && (a.ldk % 8) == 0 && (a.ldv % 8) == 0 && (a.ldo % 8) == 0, "attention: pitches must be multiples of 8");
  FO1_CHECK_ARG(((reinterpret_cast<uintptr_t>(a.q) | reinterpret_cast<uintptr_t>(a.k) | reinterpret_cast<uintptr_t>(a.v) |
                  reinterpret_cast<uintptr_t>(a.o)) & 15) == 0, "attention: q / k / v / o must be 16-byte aligned");
  if (a.n_seqs == 0 || a.total_rows <= 0) return FO1_OK;
  const int2* rowseg = reinterpret_cast<const int2*>(a.rowseg);
  if (rowseg == nullptr) {
    int2* scratch = nullptr;
    FO1_TRY(rowseg_scratch(s, (size_t)a.total_rows, &scratch));
    FO1_TRY(attention_rowseg(a.cu_seqlens, a.n_seqs, a.total_rows, reinterpret_cast<int*>(scratch), s));
    rowseg = scratch;
  }
  switch (a.head_dim) {
    case 32: return a.causal ? launch_attn_tc<32, true>(a, rowseg, s) : launch_attn_tc<32, false>(a, rowseg, s);
    case 64: return a.causal ? launch_attn_tc<64, true>(a, rowseg, s) : launch_attn_tc<64, false>(a, rowseg, s);
    case 80: return a.causal ? launch_attn_tc<80, true>(a, rowseg, s) : launch_attn_tc<80, false>(a, rowseg, s);
    case 128: return a.causal ? launch_attn_tc<128, true>(a, rowseg, s) : launch_attn_tc<128, false>(a, rowseg, s);
    default:
      set_error("attention: head_dim %d unsupported (32, 64, 80, 128)", a.head_dim);
      return FO1_ERR_UNSUPPORTED;
  }
}

}  // namespace fo1

extern "C" int fo1_attention_varlen(const fo1_attn_desc* d, void* stream) {
  using namespace fo1;
  FO1_CHECK_ARG(d != nullptr, "fo1_attention_varlen: null descriptor");
  FO1_CHECK_ARG(d->total_rows >= 0, "fo1_attention_varlen: total_rows %d", d->total_rows);
  AttnArgs a;
  a.q = static_cast<const bf16*>(d->q); a.k = static_cast<const bf16*>(d->k); a.v = static_cast<const bf16*>(d->v);
  a.o = static_cast<bf16*>(d->o);
  a.ldq = d->ldq; a.ldk = d->ldk; a.ldv = d->ldv; a.ldo = d->ldo;
  a.cu_seqlens = d->cu_seqlens; a.rowseg = nullptr; a.n_seqs = d->n_seqs; a.total_rows = d->total_rows; a.max_seqlen = d->max_seqlen;
  a.q_heads = d->q_heads; a.kv_heads = d->kv_heads; a.head_dim = d->head_dim;
  a.scale = d->scale; a.causal = d->causal; a.flops = 0.0;
  return attention_varlen(a, static_cast<cudaStream_t>(stream));
}
