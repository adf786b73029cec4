// hfre.cu -- Hybrid Fine-grained Region Encoder on sm_100a: separable-window region pooling.
//
// What the reference does (hybrid_finegrained_region_encoder.py:319-363, 230-273): up-sample aux
// levels 1..3 to level 0's grid (F.interpolate bilinear, align_corners=False), concatenate to a
// [1,3840,H/4,W/4] fp32 map (771 MB at 896^2), torchvision roi_align(7x7, sampling_ratio=-1,
// aligned=False), mean over the 49 bins; same for the primary tower's maps; concat; add a sinusoidal
// box embedding (:436-467, :55-103).
//
// What this file does instead: because every bin of a box holds the same number of samples,
// mean_{7x7}(roi_align(U))[c] = a^T U[c] b with 1-D weight vectors that depend only on the box, and
// because the up-sampling is linear and separable too, U[c] = Mh L[c] Mw^T, the whole thing is
//        out[c] = (Mh^T a)^T L[c] (Mw^T b)
// over the NATIVE-resolution bf16 level L (channels-last).  hfre_axis_weights_kernel builds the two weight vectors
// per (box, level, axis) with torchvision's exact per-sample rules.  Two interchangeable reductions follow
// (fo1_hfre_params.algo): the per-box gather (coalesced 16-byte channel vectors, fp32 FMA), which re-reads a cell once
// per covering box, and -- the default above a handful of boxes -- the map sweep, which reads every cell once and runs
// its row sums as mma.sync m16n8k16 tiles (boxes x cells, column weights split hi + lo in bf16; DESIGN.md section 4).
#include "common.cuh"

namespace fo1 {

constexpr int kMaxBatch = 32;          // images per launch: the batch descriptor travels as a kernel parameter (< 32 KB)
constexpr int kGatherThreads = 256;
constexpr int kChunk = 256;            // channels per gather block: 32 lanes x 8 bf16 (16 B) each
constexpr int kRegion = 32;            // sweep: region width in cells
constexpr int kSweepCh = 256;          // sweep: channels per CTA (4 warps x 64 channels)
constexpr int kSweepThreads = 128;
constexpr int kMmaRows = 8;            // sweep: region = kMmaRows x kRegion cells, one 16-box m-tile per pass
constexpr int kMmaSlots = 16;

struct LevelDev {
  const __nv_bfloat16* data;
  int H, W, C, upH, upW;
  float scale;
  int box_set;
  int out_off;
  int wofs;      // float offset of this level's weight records inside the image's workspace slice
  int wstride;   // floats per box record: 4 header words + H + W, rounded up to 4
  int lofs;      // int offset of this level's region box lists inside the image's list slice
  int rh, rw;    // regions (kRegion x kRegion cells) per axis
};
struct ImageDev {
  LevelDev lv[FO1_HFRE_MAX_LEVELS];
  const float* boxes[2];
  float* out;
  __nv_bfloat16* out_bf16;
  long long* acc;    // sweeps: [n_boxes][out_dim] fixed-point (2^-32) accumulators -- integer atomics commute, so the sum does
                     // not depend on the order in which the region CTAs arrive (bit-reproducible, unlike fp32 atomics)
  long long ws_ofs;  // float offset of this image's workspace slice
  long long ls_ofs;  // int offset of this image's region-list slice (after all weight records)
  int lstride;       // ints per region list: 4 header words (word 0 = count) + one kRecWords record per box
  int n_items;       // sweep work items: sum over levels of regions * ceil(C / kSweepCh)
  float pos_w, pos_h;
  int pos_box_set;
  int n_levels;
  int n_boxes;
  int n_chunks;  // sum over levels of ceil(C / kChunk)
};
struct BatchDev {
  ImageDev img[kMaxBatch];
  int n_images;
  int out_dim;
  int roi;
  int pos;
};

static_assert(sizeof(BatchDev) <= 32000, "BatchDev travels as a kernel parameter (32 KB limit on sm_70+)");

// ------------------------------------------------------------------------------------------------
// Kernel 1: per (image, box, level, axis) weight vector on the native grid.
// Sample coordinates and tap rules follow torchvision roi_align_forward_kernel_impl /
// bilinear_interpolate (aligned=False, sampling_ratio=-1): roi extent max(end-start,1); adaptive grid
// g = ceil(extent/P); sample y = start + p*bin + (i+.5)*bin/g; a sample with y < -1 or y > size
// contributes nothing; y <= 0 -> 0; y_low >= size-1 -> both taps on size-1.  Up-sampling taps follow
// ATen upsample_bilinear2d (align_corners=False): src = (in/out)*(dst+.5)-.5 clamped at 0.
// Arithmetic is written with explicit round-to-nearest ops so ptxas cannot contract it into FMAs and
// the discrete decisions (floor/ceil/skip) match the CPU kernels bit for bit.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float roi_sample_coord(float start, float bin, int p, int i, int g) {
  float t0 = __fadd_rn(start, __fmul_rn((float)p, bin));
  float t1 = __fdiv_rn(__fmul_rn(__fadd_rn((float)i, 0.5f), bin), (float)g);
  return __fadd_rn(t0, t1);
}

__global__ void __launch_bounds__(128) hfre_axis_weights_kernel(const BatchDev B, float* __restrict__ ws) {
  const ImageDev& im = B.img[blockIdx.z];
  const int box = blockIdx.x;
  const int lvl = blockIdx.y >> 1;
  const int axis = blockIdx.y & 1;  // 0: rows (y), 1: cols (x)
  if (box >= im.n_boxes || lvl >= im.n_levels) return;
  const LevelDev& L = im.lv[lvl];
  const int n_nat = axis ? L.W : L.H;
  const int n_up = axis ? L.upW : L.upH;
  const float* bx = im.boxes[L.box_set] + 4 * box;
  const float lo = axis ? bx[0] : bx[1];
  const float hi = axis ? bx[2] : bx[3];
  const int P = B.roi;

  const float start = __fmul_rn(lo, L.scale);
  const float end = __fmul_rn(hi, L.scale);
  const float extent = fmaxf(__fsub_rn(end, start), 1.0f);
  const float bin = __fdiv_rn(extent, (float)P);
  const int g = (int)ceilf(__fdiv_rn(extent, (float)P));
  const int ns = P * g;

  extern __shared__ float sm[];
  float* A = sm;            // [n_up] weights on the up-sampled axis
  // support on the up-sampled axis (samples are monotone in their index)
  const float y_first = roi_sample_coord(start, bin, 0, 0, g);
  const float y_last = roi_sample_coord(start, bin, P - 1, g - 1, g);
  int i_min = (int)floorf(fmaxf(y_first, 0.0f));
  int i_max = (int)floorf(fmaxf(y_last, 0.0f)) + 1;
  i_min = min(max(i_min, 0), n_up - 1);
  i_max = min(max(i_max, 0), n_up - 1);

  for (int r = i_min + threadIdx.x; r <= i_max; r += blockDim.x) {
    float acc = 0.0f;
    for (int p = 0; p < P; ++p) {
      for (int i = 0; i < g; ++i) {
        float y = roi_sample_coord(start, bin, p, i, g);
        const bool ok = !(y < -1.0f || y > (float)n_up);
        if (y <= 0.0f) y = 0.0f;
        int yl = (int)y, yh;
        if (yl >= n_up - 1) {
          yh = yl = n_up - 1;
          y = (float)yl;
        } else {
          yh = yl + 1;
        }
        const float ly = __fsub_rn(y, (float)yl);
        const float hy = __fsub_rn(1.0f, ly);
        if (ok) {
          if (yl == r) acc = __fadd_rn(acc, hy);
          if (yh == r) acc = __fadd_rn(acc, ly);
        }
      }
    }
    A[r] = acc;
  }
  __syncthreads();

  float* rec = ws + im.ws_ofs + L.wofs + (long long)box * L.wstride;
  int* hdr = reinterpret_cast<int*>(rec);
  float* wout = rec + 4 + (axis ? L.H : 0);
  const float norm = (float)ns;  // P * g samples per axis: mean over bins and over the bin's grid

  if (n_up == n_nat) {
    for (int r = i_min + threadIdx.x; r <= i_max; r += blockDim.x) wout[r - i_min] = __fdiv_rn(A[r], norm);
    if (threadIdx.x == 0) {
      hdr[axis * 2 + 0] = i_min;
      hdr[axis * 2 + 1] = i_max - i_min + 1;
    }
    return;
  }
  // compose with the bilinear up-sampling: native tap weights of every touched up-sampled row
  const float us = __fdiv_rn((float)n_nat, (float)n_up);
  auto src_of = [&](int i) {
    float s = __fsub_rn(__fmul_rn(us, __fadd_rn((float)i, 0.5f)), 0.5f);
    return s < 0.0f ? 0.0f : s;
  };
  const int r_min = (int)src_of(i_min);
  int r_max = (int)src_of(i_max);
  r_max = r_max + (r_max < n_nat - 1 ? 1 : 0);
  for (int r = r_min + threadIdx.x; r <= r_max; r += blockDim.x) {
    float acc = 0.0f;
    for (int i = i_min; i <= i_max; ++i) {
      const float s = src_of(i);
      const int i0 = (int)s;
      const int i1 = i0 + (i0 < n_nat - 1 ? 1 : 0);
      const float l1 = __fsub_rn(s, (float)i0);
      const float l0 = __fsub_rn(1.0f, l1);
      if (i0 == r) acc = __fadd_rn(acc, __fmul_rn(l0, A[i]));
      if (i1 == r) acc = __fadd_rn(acc, __fmul_rn(l1, A[i]));
    }
    wout[r - r_min] = __fdiv_rn(acc, norm);
  }
  if (threadIdx.x == 0) {
    hdr[axis * 2 + 0] = r_min;
    hdr[axis * 2 + 1] = r_max - r_min + 1;
  }
}

// order-independent accumulation of the region CTAs' partial sums: value * 2^32 as a 64-bit integer (|sum| < 2^31, step 2.3e-10)
__device__ __forceinline__ void acc_add(long long* p, float v) {
  atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__float2ll_rn(v * 4294967296.0f));
}

// ------------------------------------------------------------------------------------------------
// Kernel 2: out[n][d] = sinusoidal box embedding (or 0): order (cy, cx, w, h), D/4 channels each,
// interleaved sin/cos, dim_t = 10000^(2*floor(i/2)/(D/4))  (gen_sineembed_for_position :55-103).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) hfre_pos_init_kernel(const BatchDev B) {
  const ImageDev& im = B.img[blockIdx.z];
  const int box = blockIdx.y;
  if (box >= im.n_boxes) return;
  const int D = B.out_dim;
  const int q = D / 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (B.pos) {
    const float* bx = im.boxes[im.pos_box_set] + 4 * box;
    const float x1 = __fdiv_rn(bx[0], im.pos_w), y1 = __fdiv_rn(bx[1], im.pos_h);
    const float x2 = __fdiv_rn(bx[2], im.pos_w), y2 = __fdiv_rn(bx[3], im.pos_h);
    const float w = __fsub_rn(x2, x1), h = __fsub_rn(y2, y1);
    v[0] = __fadd_rn(y1, __fdiv_rn(h, 2.0f));  // cy
    v[1] = __fadd_rn(x1, __fdiv_rn(w, 2.0f));  // cx
    v[2] = w;
    v[3] = h;
  }
  float* out = im.out + (long long)box * D;
  for (int d = blockIdx.x * blockDim.x + threadIdx.x; d < D; d += gridDim.x * blockDim.x) {
    float val = 0.0f;
    if (B.pos && d < 4 * q) {
      const int part = d / q, i = d - part * q;
      const float expo = __fdiv_rn((float)(2 * (i / 2)), (float)q);
      const float dim_t = powf(10000.0f, expo);
      const float ph = __fdiv_rn(__fmul_rn(v[part], 6.283185307179586f), dim_t);
      val = (i & 1) ? cosf(ph) : sinf(ph);
    }
    out[d] = val;
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 3 (algo 1, per-box gather): one block per (image, box, level, 256-channel chunk).
// 8 warps stride over the window's rows; each lane owns 8 consecutive channels (one 16-byte load per
// cell, a warp reads 512 contiguous bytes per cell); fp32 accumulate; cross-warp reduce in smem.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kGatherThreads) hfre_gather_kernel(const BatchDev B, const float* __restrict__ ws) {
  const ImageDev& im = B.img[blockIdx.z];
  const int box = blockIdx.y;
  if (box >= im.n_boxes || (int)blockIdx.x >= im.n_chunks) return;
  // (level, chunk) of this block
  int lvl = 0, chunk = blockIdx.x;
  for (; lvl < im.n_levels; ++lvl) {
    const int nc = (im.lv[lvl].C + kChunk - 1) / kChunk;
    if (chunk < nc) break;
    chunk -= nc;
  }
  const LevelDev& L = im.lv[lvl];
  const float* rec = ws + im.ws_ofs + L.wofs + (long long)box * L.wstride;
  const int* hdr = reinterpret_cast<const int*>(rec);
  const int r0 = hdr[0], rl = hdr[1], c0 = hdr[2], cl = hdr[3];

  extern __shared__ float sm[];
  float* red = sm;                                  // [8][kChunk] (16-byte aligned for float4)
  float* wa = sm + (kGatherThreads / 32) * kChunk;  // [rl]
  float* wb = wa + L.H;                             // [cl]
  for (int i = threadIdx.x; i < rl; i += blockDim.x) wa[i] = rec[4 + i];
  for (int i = threadIdx.x; i < cl; i += blockDim.x) wb[i] = rec[4 + L.H + i];
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cbase = chunk * kChunk + lane * 8;
  const bool active = cbase < L.C;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.0f;

  if (active) {
    const long long rowpitch = (long long)L.W * L.C;
    for (int r = warp; r < rl; r += kGatherThreads / 32) {
      const float ar = wa[r];
      const __nv_bfloat16* p = L.data + (long long)(r0 + r) * rowpitch + (long long)c0 * L.C + cbase;
      int k = 0;
      for (; k + 4 <= cl; k += 4) {
        uint4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ldg_nc_v4(p + (long long)(k + u) * L.C);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float w = ar * wb[k + u];
          acc[0] = fmaf(w, bf16_lo(v[u].x), acc[0]); acc[1] = fmaf(w, bf16_hi(v[u].x), acc[1]);
          acc[2] = fmaf(w, bf16_lo(v[u].y), acc[2]); acc[3] = fmaf(w, bf16_hi(v[u].y), acc[3]);
          acc[4] = fmaf(w, bf16_lo(v[u].z), acc[4]); acc[5] = fmaf(w, bf16_hi(v[u].z), acc[5]);
          acc[6] = fmaf(w, bf16_lo(v[u].w), acc[6]); acc[7] = fmaf(w, bf16_hi(v[u].w), acc[7]);
        }
      }
      for (; k < cl; ++k) {
        const uint4 v = ldg_nc_v4(p + (long long)k * L.C);
        const float w = ar * wb[k];
        acc[0] = fmaf(w, bf16_lo(v.x), acc[0]); acc[1] = fmaf(w, bf16_hi(v.x), acc[1]);
        acc[2] = fmaf(w, bf16_lo(v.y), acc[2]); acc[3] = fmaf(w, bf16_hi(v.y), acc[3]);
        acc[4] = fmaf(w, bf16_lo(v.z), acc[4]); acc[5] = fmaf(w, bf16_hi(v.z), acc[5]);
        acc[6] = fmaf(w, bf16_lo(v.w), acc[6]); acc[7] = fmaf(w, bf16_hi(v.w), acc[7]);
      }
    }
  }
  float4* rv = reinterpret_cast<float4*>(red + warp * kChunk + lane * 8);
  rv[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
  rv[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
  __syncthreads();
  const int c = chunk * kChunk + threadIdx.x;
  if (c < L.C) {
    float s = 0.0f;
#pragma unroll
    for (int w = 0; w < kGatherThreads / 32; ++w) s += red[w * kChunk + threadIdx.x];
    float* o = im.out + (long long)box * B.out_dim + L.out_off + c;
    *o += s;  // exclusive owner of this output element (kernel 2 initialised it)
  }
}

// Region lists of the sweep below: per region, the boxes whose support meets it.  Every listed box gets its weights over
// the region's rows and columns as one contiguous 48-word record (word 0 = box id, words 4..4+kMmaRows-1 = a_y, words
// 12..43 = b_x), so a sweep pass stages its 16 boxes with ONE round of coalesced loads instead of the id -> header ->
// weights chain.
constexpr int kRecWords = 48;
static_assert(kMmaRows <= 8 && kRegion == 32, "record layout: words 4..11 = a_y, words 12..43 = b_x");
__global__ void __launch_bounds__(128) hfre_region_records_kernel(const BatchDev B, const float* __restrict__ ws, int* __restrict__ lists) {
  const ImageDev& im = B.img[blockIdx.z];
  const int lvl = blockIdx.y;
  if (lvl >= im.n_levels) return;
  const LevelDev& L = im.lv[lvl];
  const int reg = blockIdx.x;
  if (reg >= L.rh * L.rw) return;
  const int ry = reg / L.rw, rx = reg % L.rw;
  const int row0 = ry * kMmaRows, row1 = min(row0 + kMmaRows, L.H) - 1;
  const int col0 = rx * kRegion, col1 = min(col0 + kRegion, L.W) - 1;
  int* out = lists + im.ls_ofs + L.lofs + (long long)reg * im.lstride;
  __shared__ int s_count;
  if (threadIdx.x < 32) {
    int count = 0;
    for (int b0 = 0; b0 < im.n_boxes; b0 += 32) {
      const int b = b0 + threadIdx.x;
      bool hit = false;
      if (b < im.n_boxes) {
        const int* hdr = reinterpret_cast<const int*>(ws + im.ws_ofs + L.wofs + (long long)b * L.wstride);
        const int r0 = hdr[0], r1 = hdr[0] + hdr[1] - 1, c0 = hdr[2], c1 = hdr[2] + hdr[3] - 1;
        hit = r0 <= row1 && r1 >= row0 && c0 <= col1 && c1 >= col0;
      }
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (hit) out[4 + (count + __popc(m & ((1u << threadIdx.x) - 1u))) * kRecWords] = b;
      count += __popc(m);
    }
    if (threadIdx.x == 0) { out[0] = count; s_count = count; }
  }
  __syncthreads();   // block-scope visibility of the ids written above
  const int count = s_count;
  float* fout = reinterpret_cast<float*>(out);
  for (int i = threadIdx.x; i < count * (kMmaRows + kRegion); i += blockDim.x) {
    const int sl = i / (kMmaRows + kRegion), j = i % (kMmaRows + kRegion);
    const int axis = j >= kMmaRows, k = axis ? j - kMmaRows : j;
    const int b = out[4 + sl * kRecWords];
    const float* rec = ws + im.ws_ofs + L.wofs + (long long)b * L.wstride;
    const int* hdr = reinterpret_cast<const int*>(rec);
    const int start = hdr[axis * 2], len = hdr[axis * 2 + 1];
    const int idx = (axis ? col0 : row0) + k - start;
    fout[4 + sl * kRecWords + (axis ? 12 + k : 4 + k)] = (idx >= 0 && idx < len) ? rec[4 + (axis ? L.H : 0) + idx] : 0.0f;
  }
}

// ------------------------------------------------------------------------------------------------
// Kernel 3' (algo 3, map sweep on the tensor pipe).  The per-box gather re-reads every cell once per covering box (~8x
// the unique bytes at 100 boxes/image, L2-bound); the sweep inverts the loops so that a CTA reads each cell of its region
// once.  At C2's box density every cell is covered by ~7 boxes, i.e. ~7.5 FLOP per loaded byte: with the bf16 -> fp32
// unpacking a sweep on the FMA pipe is issue-bound at ~1/8 of the HBM roofline (profiles/: FMA pipe 26 %, 488 M warp
// instructions for 1.3 GB).  The reduction is a contraction,
//     out[box][c] += sum_y a_y[box] * ( sum_x b_x[box] * L[y][x][c] ),
// so the inner sum over a region row runs as mma.sync m16n8k16 (A = b_x of 16 boxes, B = 16 cells x 8 channels of
// the bf16 map, fp32 accumulate) and only the per-row scaling by a_y stays on the FMA pipe (1 FMA per 32 MACs).
// The fp32 weights are fed as hi + lo bf16 halves (two MMAs): the map is bf16 already, so products are exact and
// the weights keep 16 mantissa bits -- inside the 1e-3 parity budget with three orders of margin.
// Work split: CTA = (level, 8 x 32 cell region, 256 channels), warp = 64 channels, a pass accumulates 16 boxes (one
// m-tile; regions with more boxes take further passes whose rows come from L2 -- 8-row regions keep the footprint of
// all resident CTAs below the L2 size).  A fragments depend on the boxes only and are built once per pass from the
// region's weight records (hfre_region_records_kernel).  Every region row is copied ONCE per pass into a per-warp
// cp.async ring (3 rows, two in flight behind the one being reduced; 16-byte chunks XOR-swizzled by cell) and its
// B fragments are taken with ldmatrix.trans.  The partial sums of the pass leave through shared memory (aliasing the
// ring) as coalesced fp32 reductions into out[box][channel].
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// w0, w1 -> packed bf16 pairs of their high parts and of the remainders
__device__ __forceinline__ void split_pair(float w0, float w1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16_rn(w0), h1 = __float2bfloat16_rn(w1);
  hi = pack_bf16(__bfloat162float(h0), __bfloat162float(h1));
  lo = pack_bf16(w0 - __bfloat162float(h0), w1 - __bfloat162float(h1));
}

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst_smem, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;  // src-size 0 -> 16 bytes of zeros
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async16_plain(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
constexpr int kMmaStages = 3;                                   // per-warp ring of region rows (cp.async)
constexpr int kMmaRowBytes = kRegion * 128;                     // 32 cells x 64 channels x 2 B
constexpr int kMmaRingBytes = (kSweepThreads / 32) * kMmaStages * kMmaRowBytes;
constexpr int kMmaAccPitch = kSweepCh + 4;                      // floats; the flush staging aliases the ring
constexpr int kMmaSmemBytes = kMmaRingBytes + kMmaSlots * (kMmaRows + kRegion) * 4 + kMmaSlots * 4 + 16;
static_assert(kMmaSlots * kMmaAccPitch * 4 <= kMmaRingBytes, "flush staging must fit in the ring it aliases");

__global__ void __launch_bounds__(kSweepThreads, 4) hfre_sweep_mma_kernel(const BatchDev B, const float* __restrict__ ws, const int* __restrict__ lists) {
  const ImageDev& im = B.img[blockIdx.z];
  if ((int)blockIdx.x >= im.n_items) return;
  int lvl = 0, item = blockIdx.x;
  for (; lvl < im.n_levels; ++lvl) {
    const int n = im.lv[lvl].rh * im.lv[lvl].rw * ((im.lv[lvl].C + kSweepCh - 1) / kSweepCh);
    if (item < n) break;
    item -= n;
  }
  const LevelDev& L = im.lv[lvl];
  const int n_reg = L.rh * L.rw;
  const int cgroup = item / n_reg, reg = item % n_reg;
  const int* list = lists + im.ls_ofs + L.lofs + (long long)reg * im.lstride;
  const int n_list = list[0];
  if (n_list == 0) return;  // no box touches this region: its cells are never read
  const int ry = reg / L.rw, rx = reg % L.rw;
  const int row0 = ry * kMmaRows, col0 = rx * kRegion;

  extern __shared__ __align__(128) uint8_t s_dyn[];
  float* s_acc = reinterpret_cast<float*>(s_dyn);                                   // [kMmaSlots][kMmaAccPitch], aliases the ring
  float (*s_wa)[kMmaRows] = reinterpret_cast<float (*)[kMmaRows]>(s_dyn + kMmaRingBytes);
  float (*s_wb)[kRegion] = reinterpret_cast<float (*)[kRegion]>(s_dyn + kMmaRingBytes + kMmaSlots * kMmaRows * 4);
  int* s_box = reinterpret_cast<int*>(s_dyn + kMmaRingBytes + kMmaSlots * (kMmaRows + kRegion) * 4);
  unsigned* s_mask = reinterpret_cast<unsigned*>(s_box + kMmaSlots);                // [0] rows, [1] column halves

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  const int cbase = cgroup * kSweepCh + warp * 64;        // this warp's 64 channels
  const long long rowpitch = (long long)L.W * L.C;
  const uint32_t ring = (uint32_t)__cvta_generic_to_shared(s_dyn) + warp * kMmaStages * kMmaRowBytes;
  // cp.async: instruction i moves 16-byte chunk (cell = 4i + lane/8, channels 8*(lane%8) ..); 16-byte chunks of a cell row
  // are XOR-swizzled by (cell & 7) so the transposing ldmatrix reads below are bank-conflict-free
  const int cp_cell = lane >> 3, cp_chunk = lane & 7;
  const bool cp_ch_ok = cbase + cp_chunk * 8 < L.C;       // C % 8 == 0
  // everything about the 8 copies of a row that does not depend on the row is computed once: source column pointer
  // (cell i*4 + cp_cell is i * 4C elements further), validity bits, the two swizzled destinations (even / odd i)
  const __nv_bfloat16* cp_src = L.data + (cp_ch_ok ? cbase + cp_chunk * 8 : 0) + (long long)min(col0 + cp_cell, L.W - 1) * L.C;
  const long long cp_step = 4LL * L.C;
  unsigned cp_ok = 0u;
#pragma unroll
  for (int i = 0; i < 8; ++i) cp_ok |= (cp_ch_ok && col0 + i * 4 + cp_cell < L.W) ? (1u << i) : 0u;
  const uint32_t cp_dst_even = ring + cp_cell * 128 + ((cp_chunk ^ cp_cell) << 4);
  const uint32_t cp_dst_odd = ring + (cp_cell + 4) * 128 + ((cp_chunk ^ (cp_cell + 4)) << 4);
  // ldmatrix.x4.trans: lane -> row (cell (m&1)*8 + r of the 16-cell k-step) of matrix m = lane/8; matrices 0,1 = n-tile 2p, 2,3 = 2p+1
  const int lm_cell = ((lane >> 3) & 1) * 8 + (lane & 7), lm_half = lane >> 4;

  for (int base = 0; base < n_list; base += kMmaSlots) {
    const int ns = min(kMmaSlots, n_list - base);
    const int* recs = list + 4 + (long long)base * kRecWords;
    if (threadIdx.x < kMmaSlots) s_box[threadIdx.x] = threadIdx.x < ns ? recs[threadIdx.x * kRecWords] : -1;
    if (threadIdx.x < 2) s_mask[threadIdx.x] = 0u;
    __syncthreads();
    {
      // 8 threads per slot: words 4..11 of the record are a_y, 12..43 are b_x (five strided words per thread)
      static_assert(kSweepThreads == kMmaSlots * 8 && kMmaRows == 8, "staging layout");
      const int sl = threadIdx.x >> 3, q = threadIdx.x & 7;
      const int* rec = recs + sl * kRecWords + 4 + q;
      unsigned rbits = 0u, cbits = 0u;
      float w[5];
#pragma unroll
      for (int r = 0; r < 5; ++r) w[r] = sl < ns ? __int_as_float(rec[8 * r]) : 0.0f;
      s_wa[sl][q] = w[0];
      if (w[0] != 0.0f) rbits = 1u << q;
#pragma unroll
      for (int r = 1; r < 5; ++r) {
        s_wb[sl][q + 8 * (r - 1)] = w[r];
        if (w[r] != 0.0f) cbits |= 1u << ((r - 1) >> 1);
      }
      rbits = __reduce_or_sync(0xffffffffu, rbits);
      cbits = __reduce_or_sync(0xffffffffu, cbits);
      if (lane == 0) { atomicOr(&s_mask[0], rbits); atomicOr(&s_mask[1], cbits); }
    }
    __syncthreads();

    // A fragments: rows = boxes (g, g+8), k-slots (2t, 2t+1 | 2t+8, 2t+9) = columns of the half; built once per pass
    uint32_t ahi[2][4], alo[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float* wb = &s_wb[g + 8 * h][ks * 16 + 2 * t];
        split_pair(wb[0], wb[1], ahi[ks][h], alo[ks][h]);
        split_pair(wb[8], wb[9], ahi[ks][2 + h], alo[ks][2 + h]);
      }
    float acc[8][4];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e][0] = acc[e][1] = acc[e][2] = acc[e][3] = 0.f;

    const unsigned rows_any = s_mask[0];      // rows beyond the map carry zero weights and are never selected
    const unsigned cols_any = s_mask[1];
    unsigned pending = rows_any, todo = rows_any;
    uint32_t st_issue = 0, st_done = 0;       // ring stage offsets (bytes) of the next row to fetch / to reduce
    auto issue_row = [&]() {                  // next active row -> next ring stage (always commits a group)
      if (pending) {
        const int y = __ffs(pending) - 1;
        pending &= pending - 1;
        const __nv_bfloat16* prow = cp_src + (long long)(row0 + y) * rowpitch;
        if (cp_ok == 0xffu) {                                // region and channel slice fully on the map: no predication
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (!((cols_any >> (i >> 2)) & 1u)) continue;  // column half without weights: neither loaded nor multiplied
            cp_async16_plain(((i & 1) ? cp_dst_odd + (i - 1) * 512 : cp_dst_even + i * 512) + st_issue, prow + i * cp_step);
          }
        } else {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (!((cols_any >> (i >> 2)) & 1u)) continue;
            const bool ok = (cp_ok >> i) & 1u;             // off-map cells / channels: zero-filled, source pointer stays in range
            cp_async16_zfill(((i & 1) ? cp_dst_odd + (i - 1) * 512 : cp_dst_even + i * 512) + st_issue, ok ? prow + i * cp_step : prow, ok);
          }
        }
        st_issue = (st_issue == (kMmaStages - 1) * kMmaRowBytes) ? 0u : st_issue + kMmaRowBytes;
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue_row();
    issue_row();
    while (todo) {
      const int y = __ffs(todo) - 1;
      todo &= todo - 1;
      issue_row();                                            // two rows stay in flight behind the one being reduced
      asm volatile("cp.async.wait_group 2;" ::: "memory");
      __syncwarp();
      const uint32_t stage = ring + st_done;
      const float wa0 = s_wa[g][y], wa1 = s_wa[g + 8][y];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        float tq[2][4];   // row sums of the pair's two n-tiles; the hi and lo weight halves accumulate into the same registers
#pragma unroll
        for (int q = 0; q < 2; ++q) { tq[q][0] = tq[q][1] = tq[q][2] = tq[q][3] = 0.f; }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {
          if (!((cols_any >> ks) & 1u)) continue;   // warp-uniform
          const int cell = ks * 16 + lm_cell;
          uint32_t bf[4];
          ldsm_x4_t(bf, stage + cell * 128 + (((2 * p + lm_half) ^ (cell & 7)) << 4));
          mma_bf16_16816(tq[0], ahi[ks], bf[0], bf[1]); mma_bf16_16816(tq[1], ahi[ks], bf[2], bf[3]);
          mma_bf16_16816(tq[0], alo[ks], bf[0], bf[1]); mma_bf16_16816(tq[1], alo[ks], bf[2], bf[3]);
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          float* a4 = acc[2 * p + q];
          a4[0] = fmaf(wa0, tq[q][0], a4[0]); a4[1] = fmaf(wa0, tq[q][1], a4[1]);
          a4[2] = fmaf(wa1, tq[q][2], a4[2]); a4[3] = fmaf(wa1, tq[q][3], a4[3]);
        }
      }
      __syncwarp();                                           // the stage may be refilled by the next issue_row()
      st_done = (st_done == (kMmaStages - 1) * kMmaRowBytes) ? 0u : st_done + kMmaRowBytes;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();                                          // every warp is done with its ring: reuse it as the flush staging
    // accumulator columns (2t, 2t+1) of n-tile e are channels e*8 + 2t, +1 of the warp's 64
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      *reinterpret_cast<float2*>(&s_acc[g * kMmaAccPitch + warp * 64 + e * 8 + 2 * t]) = make_float2(acc[e][0], acc[e][1]);
      *reinterpret_cast<float2*>(&s_acc[(g + 8) * kMmaAccPitch + warp * 64 + e * 8 + 2 * t]) = make_float2(acc[e][2], acc[e][3]);
    }
    __syncthreads();
    {
      // thread -> channels (tid, tid + 128) of every box of the pass: one row pointer per box, two coalesced reductions
      const int c0 = cgroup * kSweepCh + threadIdx.x;
      long long* obase = im.acc + L.out_off + c0;
      for (int sl = 0; sl < ns; ++sl) {
        long long* orow = obase + (long long)s_box[sl] * B.out_dim;
        if (c0 < L.C) acc_add(orow, s_acc[sl * kMmaAccPitch + threadIdx.x]);
        if (c0 + kSweepThreads < L.C) acc_add(orow + kSweepThreads, s_acc[sl * kMmaAccPitch + threadIdx.x + kSweepThreads]);
      }
    }
    __syncthreads();
  }
}

// Kernel 4: finish -- sweeps: out = box embedding (already in out) + pooled feature (the fixed-point sum, rounded to fp32 once:
// the reference adds the embedding to the finished feature, hybrid_finegrained_region_encoder.py:464-467); then the optional
// bf16 copy (the reference casts to the tower dtype before mm_projector_aux, omchat_qwen2_5_vl.py:106).
__global__ void __launch_bounds__(256) hfre_finish_kernel(const BatchDev B, int from_acc) {
  const ImageDev& im = B.img[blockIdx.z];
  if (!from_acc && im.out_bf16 == nullptr) return;
  const long long n = (long long)im.n_boxes * B.out_dim;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v = im.out[i];
    if (from_acc) {
      v = __fadd_rn((float)((double)im.acc[i] * (1.0 / 4294967296.0)), v);
      im.out[i] = v;
    }
    if (im.out_bf16 != nullptr) im.out_bf16[i] = __float2bfloat16_rn(v);
  }
}

// ---------------------------------------------------------------------------------------------- host
static int level_wstride(const fo1_hfre_level& l) { return (4 + l.H + l.W + 3) & ~3; }

static size_t image_ws_floats(const fo1_hfre_image& im) {
  size_t f = 0;
  for (int l = 0; l < im.n_levels; ++l) f += (size_t)im.n_boxes * level_wstride(im.levels[l]);
  return f;
}
static int record_stride(int n_boxes) { return 4 + n_boxes * kRecWords; }             // count + 48-word records
static size_t image_list_ints(const fo1_hfre_image& im) {
  size_t n = 0;
  for (int l = 0; l < im.n_levels; ++l)
    n += (size_t)ceil_div(im.levels[l].H, kMmaRows) * ceil_div(im.levels[l].W, kRegion) * record_stride(im.n_boxes);
  return n;
}

}  // namespace fo1

using namespace fo1;

static size_t acc_bytes(const fo1_hfre_image* images, int n_images, const fo1_hfre_params* p) {
  size_t n = 0;
  for (int i = 0; i < n_images; ++i) n += (size_t)(images[i].n_boxes > 0 ? images[i].n_boxes : 0) * (size_t)(p ? p->out_dim : 0);
  return n * sizeof(long long);
}

extern "C" size_t fo1_hfre_workspace_bytes(const fo1_hfre_image* images, int32_t n_images, const fo1_hfre_params* p) {
  size_t f = 0;
  for (int i = 0; i < n_images; ++i) f += image_ws_floats(images[i]) + image_list_ints(images[i]);
  return ((f * sizeof(float) + 255) & ~(size_t)255) + acc_bytes(images, n_images, p) + 256;
}

extern "C" int fo1_hfre_forward(const fo1_hfre_image* images, int32_t n_images, const fo1_hfre_params* p,
                                void* workspace, size_t workspace_bytes, void* stream_) {
  FO1_CHECK_ARG(images && p && n_images >= 0, "fo1_hfre_forward: null argument");
  if (n_images == 0) return FO1_OK;
  FO1_CHECK_ARG(p->roi_size >= 1 && p->roi_size <= 32, "fo1_hfre_forward: roi_size %d unsupported", p->roi_size);
  FO1_CHECK_ARG(p->out_dim > 0 && p->out_dim % 4 == 0, "fo1_hfre_forward: out_dim %d must be a positive multiple of 4", p->out_dim);
  FO1_CHECK_ARG(p->algo == 0 || p->algo == 1 || p->algo == 3, "fo1_hfre_forward: algo %d not available (0 auto, 1 gather, 3 sweep)", p->algo);
  const size_t need = fo1_hfre_workspace_bytes(images, n_images, p);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("fo1_hfre_forward: workspace %zu B < required %zu B", workspace_bytes, need);
    return FO1_ERR_WORKSPACE;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  float* ws = static_cast<float*>(workspace);
  size_t total_w = 0;
  for (int i = 0; i < n_images; ++i) total_w += image_ws_floats(images[i]);
  int* lists = reinterpret_cast<int*>(ws + total_w);   // region box lists live after all weight records
  size_t ls_ofs = 0;
  size_t total_f = 0;
  for (int i = 0; i < n_images; ++i) total_f += image_ws_floats(images[i]) + image_list_ints(images[i]);
  long long* acc_base = reinterpret_cast<long long*>(static_cast<char*>(workspace) + ((total_f * sizeof(float) + 255) & ~(size_t)255));
  size_t acc_ofs = 0;
  bool acc_zeroed = false;

  size_t ws_ofs = 0;
  for (int base = 0; base < n_images; base += kMaxBatch) {
    BatchDev B;
    memset(&B, 0, sizeof(B));
    B.n_images = (n_images - base < kMaxBatch) ? n_images - base : kMaxBatch;
    B.out_dim = p->out_dim;
    B.roi = p->roi_size;
    B.pos = p->apply_pos_embed ? 1 : 0;
    int batch_boxes = 0;
    for (int i = 0; i < B.n_images; ++i) batch_boxes += images[base + i].n_boxes > 0 ? images[base + i].n_boxes : 0;
    // algo 0: the sweep wins as soon as boxes overlap (its traffic is the union of the windows, the gather's their sum)
    const bool sweep = p->algo == 3 || (p->algo == 0 && batch_boxes >= 8 * B.n_images);
    int max_boxes = 0, max_levels = 0, max_chunks = 0, max_up = 0, max_hw = 0, max_items = 0, max_regions = 0;
    for (int i = 0; i < B.n_images; ++i) {
      const fo1_hfre_image& src = images[base + i];
      ImageDev& d = B.img[i];
      FO1_CHECK_ARG(src.n_levels >= 1 && src.n_levels <= FO1_HFRE_MAX_LEVELS, "image %d: n_levels %d out of range", base + i, src.n_levels);
      FO1_CHECK_ARG(src.n_boxes >= 0, "image %d: negative n_boxes", base + i);
      FO1_CHECK_ARG(src.n_boxes == 0 || (src.boxes_aux && src.boxes_vt && src.out), "image %d: null boxes/out", base + i);
      d.n_levels = src.n_levels;
      d.n_boxes = src.n_boxes;
      d.boxes[0] = src.boxes_aux;
      d.boxes[1] = src.boxes_vt;
      d.out = src.out;
      d.out_bf16 = static_cast<__nv_bfloat16*>(src.out_bf16);
      d.acc = acc_base + acc_ofs;
      acc_ofs += (size_t)(src.n_boxes > 0 ? src.n_boxes : 0) * (size_t)p->out_dim;
      d.pos_w = src.pos_img_w;
      d.pos_h = src.pos_img_h;
      d.pos_box_set = src.pos_box_set ? 1 : 0;
      d.ws_ofs = (long long)ws_ofs;
      int wofs = 0, chunks = 0, lofs = 0, items = 0;
      d.ls_ofs = (long long)ls_ofs;
      d.lstride = record_stride(src.n_boxes);
      for (int l = 0; l < src.n_levels; ++l) {
        const fo1_hfre_level& sl = src.levels[l];
        FO1_CHECK_ARG(sl.data != nullptr && sl.H > 0 && sl.W > 0 && sl.C > 0, "image %d level %d: bad shape", base + i, l);
        FO1_CHECK_ARG(sl.C % 8 == 0, "image %d level %d: C=%d must be a multiple of 8", base + i, l, sl.C);
        FO1_CHECK_ARG((reinterpret_cast<uintptr_t>(sl.data) & 15) == 0, "image %d level %d: data not 16-byte aligned", base + i, l);
        FO1_CHECK_ARG(sl.up_H >= sl.H && sl.up_W >= sl.W, "image %d level %d: up-sampled grid smaller than native", base + i, l);
        FO1_CHECK_ARG(sl.out_offset >= 0 && sl.out_offset + sl.C <= p->out_dim, "image %d level %d: channels [%d,%d) exceed out_dim %d", base + i, l, sl.out_offset, sl.out_offset + sl.C, p->out_dim);
        LevelDev& dl = d.lv[l];
        dl.data = static_cast<const __nv_bfloat16*>(sl.data);
        dl.H = sl.H; dl.W = sl.W; dl.C = sl.C; dl.upH = sl.up_H; dl.upW = sl.up_W;
        dl.scale = sl.spatial_scale;
        dl.box_set = sl.box_set ? 1 : 0;
        dl.out_off = sl.out_offset;
        dl.wofs = wofs;
        dl.wstride = level_wstride(sl);
        wofs += src.n_boxes * dl.wstride;
        chunks += ceil_div(sl.C, kChunk);
        dl.rh = ceil_div(sl.H, kMmaRows); dl.rw = ceil_div(sl.W, kRegion);
        dl.lofs = lofs;
        lofs += dl.rh * dl.rw * d.lstride;
        items += dl.rh * dl.rw * ceil_div(sl.C, kSweepCh);
        max_regions = max_regions > dl.rh * dl.rw ? max_regions : dl.rh * dl.rw;
        max_up = max_up > sl.up_H ? max_up : sl.up_H;
        max_up = max_up > sl.up_W ? max_up : sl.up_W;
        max_hw = max_hw > sl.H + sl.W ? max_hw : sl.H + sl.W;
      }
      d.n_chunks = chunks;
      d.n_items = items;
      max_items = max_items > items ? max_items : items;
      ws_ofs += (size_t)wofs;
      ls_ofs += (size_t)lofs;
      max_boxes = max_boxes > src.n_boxes ? max_boxes : src.n_boxes;
      max_levels = max_levels > src.n_levels ? max_levels : src.n_levels;
      max_chunks = max_chunks > chunks ? max_chunks : chunks;
    }
    if (max_boxes == 0) continue;
    {
      dim3 grid(max_boxes, max_levels * 2, B.n_images);
      ProfScope prof("hfre_weights", 0.0, 0.0, stream);
      hfre_axis_weights_kernel<<<grid, 128, (size_t)max_up * sizeof(float), stream>>>(B, ws);
      FO1_LAUNCH_CHECK();
    }
    {
      dim3 grid(ceil_div(p->out_dim, 256 * 4), max_boxes, B.n_images);
      hfre_pos_init_kernel<<<grid, 256, 0, stream>>>(B);
      FO1_LAUNCH_CHECK();
    }
    if (sweep) {
      if (!acc_zeroed) {   // one memset for every image of the call
        FO1_CUDA(cudaMemsetAsync(acc_base, 0, acc_bytes(images, n_images, p), stream));
        acc_zeroed = true;
      }
      {
        dim3 grid(max_regions, max_levels, B.n_images);
        hfre_region_records_kernel<<<grid, 128, 0, stream>>>(B, ws, lists);
        FO1_LAUNCH_CHECK();
      }
      dim3 grid(max_items, 1, B.n_images);
      ProfScope prof("hfre_sweep_mma", 0.0, 0.0, stream);
      static bool attr_set = false;
      if (!attr_set) {
        FO1_CUDA(cudaFuncSetAttribute(hfre_sweep_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMmaSmemBytes));
        attr_set = true;
      }
      hfre_sweep_mma_kernel<<<grid, kSweepThreads, kMmaSmemBytes, stream>>>(B, ws, lists);
      FO1_LAUNCH_CHECK();
    } else {
      dim3 grid(max_chunks, max_boxes, B.n_images);
      const size_t smem = ((size_t)max_hw + (kGatherThreads / 32) * kChunk) * sizeof(float);
      ProfScope prof("hfre_gather", 0.0, 0.0, stream);
      hfre_gather_kernel<<<grid, kGatherThreads, smem, stream>>>(B, ws);
      FO1_LAUNCH_CHECK();
    }
    bool any_bf16 = false;
    for (int i = 0; i < B.n_images; ++i) any_bf16 |= (B.img[i].out_bf16 != nullptr);
    if (any_bf16 || sweep) {
      dim3 grid(ceil_div(max_boxes * p->out_dim, 256 * 8), 1, B.n_images);
      hfre_finish_kernel<<<grid, 256, 0, stream>>>(B, sweep ? 1 : 0);
      FO1_LAUNCH_CHECK();
    }
  }
  return FO1_OK;
}
