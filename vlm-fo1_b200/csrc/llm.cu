// llm.cu -- Qwen2.5 decoder on sm_100a: embedding splice, M-RoPE bookkeeping, varlen prefill, device-resident
// greedy decode with a static K/V cache.
//
// Reference: OmChatQwen25VLForCausalLM.forward + prepare_inputs_labels_for_qwen2_5_vl_multimodal
// (omchat_qwen2_5_vl.py:135-532), Qwen2_5_VLModel / DecoderLayer / Attention / MLP / RMSNorm
// (modeling_qwen2_5_vl.py:1126-1242, 1014-1095, 738-802, 627-640, 126-140), get_rope_index (:1546-1721),
// the decode position rule (:1848-1860) and HF's greedy loop with KeywordsStoppingCriteria (mm_utils.py:137-181).
// B200-first differences: all sequences of the batch run packed (varlen), no padding tokens exist; K/V live
// in one static [layer][seq][cap][kv] cache written by the prefill and appended in place by each decode
// step (the reference torch.cat's a DynamicCache per layer per step); argmax, stop-token test and all loop
// state stay on the device, the host only enqueues kernels (no per-token sync); lm_head runs on the last
// prompt position only.
#include <algorithm>

#include "decode_mega.cuh"

namespace fo1 {

// ------------------------------------------------------------------------------------------ kernels
// inputs_embeds rows from three sources
__global__ void __launch_bounds__(256) build_embeds_kernel(const int* __restrict__ kind, const int* __restrict__ index,
                                                           const bf16* __restrict__ table, const bf16* __restrict__ img,
                                                           const bf16* __restrict__ reg, bf16* __restrict__ out, int H) {
  const int r = blockIdx.x;
  const int k = kind[r];
  const bf16* src = (k == 0 ? table : (k == 1 ? img : reg)) + (long long)index[r] * H;
  bf16* dst = out + (long long)r * H;
  for (int c = threadIdx.x * 8; c < H; c += blockDim.x * 8) *reinterpret_cast<uint4*>(dst + c) = *reinterpret_cast<const uint4*>(src + c);
}

// x[b] = table[tok[b]]
__global__ void __launch_bounds__(256) embed_tokens_kernel(const int* __restrict__ tok, const bf16* __restrict__ table,
                                                           bf16* __restrict__ out, int H) {
  griddep_launch();
  griddep_wait();
  const bf16* src = table + (long long)tok[blockIdx.x] * H;
  bf16* dst = out + (long long)blockIdx.x * H;
  for (int c = threadIdx.x * 8; c < H; c += blockDim.x * 8) *reinterpret_cast<uint4*>(dst + c) = *reinterpret_cast<const uint4*>(src + c);
}

// prefill: copy the rotated K and V of packed row r into the cache slot (seq[r], t[r])
__global__ void __launch_bounds__(128) kv_store_kernel(const bf16* __restrict__ qkv, long long ld, int q_dim, int kv_dim,
                                                       const int* __restrict__ row_seq, const int* __restrict__ row_t,
                                                       bf16* __restrict__ kc, bf16* __restrict__ vc, int cap) {
  const int r = blockIdx.x;
  const long long slot = ((long long)row_seq[r] * cap + row_t[r]) * kv_dim;
  const bf16* kp = qkv + (long long)r * ld + q_dim;
  for (int c = threadIdx.x * 8; c < kv_dim; c += blockDim.x * 8) {
    *reinterpret_cast<uint4*>(kc + slot + c) = *reinterpret_cast<const uint4*>(kp + c);
    *reinterpret_cast<uint4*>(vc + slot + c) = *reinterpret_cast<const uint4*>(kp + kv_dim + c);
  }
}
// Single-query GQA attention over the cache, split over the sequence (flash-decoding) and run on the tensor pipe:
// one block per (sequence, kv head, split).  The G <= 8 query heads of the kv head are the rows of an m16n8k16 tile
// (rows G..15 are zero), so K and V are read ONCE per kv head instead of once per query head.  Every warp owns
// 16-key tiles of the split and streams them through a private cp.async ring (3 tiles = 24 KB, two in flight behind
// the one being reduced; 16-byte chunks XOR-swizzled by key) -- the load -> use chain of a register-fed version left
// a warp with one tile in flight and the kernel at 1.3 TB/s.  S = Q.K^T takes its B fragments with ldmatrix, P.V with
// ldmatrix.trans; the block merges its warps' (m, l, acc) and writes one un-normalised partial per (head, split);
// decode_attn_combine_kernel merges the splits.
constexpr int kDecSplits = 8;   // most key splits per (sequence, kv head); the launch uses gridDim.z <= kDecSplits of them
constexpr int kDecWarps = 4;
constexpr int kDecStages = 3;
constexpr int kDecTileBytes = 16 * 256 * 2;                      // 16 keys x (K row 256 B + V row 256 B)
constexpr int kDecRingBytes = kDecWarps * kDecStages * kDecTileBytes;
constexpr int kDecSmemBytes = kDecRingBytes;                     // the warp merge staging aliases the ring
__device__ __forceinline__ void mma_m16n8k16(float (&c)[4], uint32_t a0, uint32_t a2, uint32_t b0, uint32_t b1) {
  // rows 8..15 of A (a1, a3) are zero: only the G query heads in rows 0..7 carry data
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%5}, {%7,%8}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(0u), "r"(a2), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2_bf16(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ void dec_cp16(uint32_t dst, const void* src, bool valid) {
  const int sz = valid ? 16 : 0;  // src-size 0 -> 16 bytes of zeros
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void dec_ldsm(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void dec_ldsm_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__global__ void __launch_bounds__(kDecWarps * 32) decode_attn_kernel(const bf16* __restrict__ q, long long ldq, const bf16* __restrict__ kc,
                                                                     const bf16* __restrict__ vc, const int* __restrict__ cache_len, int cap,
                                                                     int kv_heads, int G, float* __restrict__ part, float scale) {
  constexpr int HD = 128;
  extern __shared__ __align__(128) uint8_t dec_smem[];
  const int b = blockIdx.x, kvh = blockIdx.y, sp = blockIdx.z;
  griddep_launch();
  griddep_wait();
  const int n = cache_len[b] + 1;  // the step's own K/V was appended at index cache_len[b]
  const int n_splits = gridDim.z;
  const int chunk = ((n + n_splits - 1) / n_splits + 15) & ~15;
  const int t_begin = sp * chunk, t_end = min(n, t_begin + chunk);
  const int kv_dim = kv_heads * HD;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;
  // Q fragments (A operand, rows = heads): a0 = dims (16 ks + 2t, +1), a2 = dims (16 ks + 8 + 2t, +1) of head g
  uint32_t qa[8][2];
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) { qa[ks][0] = 0u; qa[ks][1] = 0u; }
  if (g < G) {
    const bf16* qp = q + (long long)b * ldq + (long long)(kvh * G + g) * HD + 2 * t;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      qa[ks][0] = *reinterpret_cast<const uint32_t*>(qp + ks * 16);
      qa[ks][1] = *reinterpret_cast<const uint32_t*>(qp + ks * 16 + 8);
    }
  }
  const float sc = scale * 1.4426950408889634f;
  float m = -INFINITY, l = 0.f, o[16][4];
#pragma unroll
  for (int j = 0; j < 16; ++j) { o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f; }

  const uint32_t ring = (uint32_t)__cvta_generic_to_shared(dec_smem) + w * kDecStages * kDecTileBytes;
  // copy plan: instruction i moves chunk (key = 2i + lane/16, 16-byte chunk lane%16) of the K half and of the V half
  const int cp_key = lane >> 4, cp_chunk = lane & 15;
  const bf16* kbase = kc + (long long)b * cap * kv_dim + kvh * HD + cp_chunk * 8;
  const bf16* vbase = vc + (long long)b * cap * kv_dim + kvh * HD + cp_chunk * 8;
  int t_issue = t_begin + w * 16;
  uint32_t st_issue = 0, st_done = 0;
  auto issue_tile = [&]() {
    if (t_issue < t_end) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int key = 2 * i + cp_key, tok = t_issue + key;
        const bool ok = tok < t_end;                          // keys beyond the split: zero rows (their scores are masked)
        const long long off = (long long)(ok ? tok : t_begin) * kv_dim;
        const uint32_t dst = ring + st_issue + key * 256 + ((cp_chunk ^ (key & 7)) << 4);
        dec_cp16(dst, kbase + off, ok);
        dec_cp16(dst + 16 * 256, vbase + off, ok);
      }
      t_issue += kDecWarps * 16;
      st_issue = (st_issue == (kDecStages - 1) * kDecTileBytes) ? 0u : st_issue + kDecTileBytes;
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  issue_tile();
  issue_tile();
  // ldmatrix lane roles: S: matrix m = lane/8 -> (keys (m/2)*8 + r, chunk 2 ks + (m&1)); PV (trans): (keys (m&1)*8 + r, chunk c + m/2)
  const int lr = lane & 7, lm = lane >> 3;
  for (int t0 = t_begin + w * 16; t0 < t_end; t0 += kDecWarps * 16) {
    issue_tile();
    asm volatile("cp.async.wait_group 2;" ::: "memory");
    __syncwarp();
    const uint32_t kt = ring + st_done, vt = kt + 16 * 256;
    float s[2][4];
#pragma unroll
    for (int i = 0; i < 2; ++i) { s[i][0] = s[i][1] = s[i][2] = s[i][3] = 0.f; }
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      uint32_t bk[4];
      const int key = (lm >> 1) * 8 + lr;
      dec_ldsm(bk, kt + key * 256 + (((2 * ks + (lm & 1)) ^ (key & 7)) << 4));
      mma_m16n8k16(s[0], qa[ks][0], qa[ks][1], bk[0], bk[1]);
      mma_m16n8k16(s[1], qa[ks][0], qa[ks][1], bk[2], bk[3]);
    }
    float tmax = -INFINITY;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        s[i][e] = (t0 + i * 8 + 2 * t + e < t_end) ? s[i][e] * sc : -INFINITY;
        tmax = fmaxf(tmax, s[i][e]);
      }
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 1));
    tmax = fmaxf(tmax, __shfl_xor_sync(0xffffffffu, tmax, 2));
    const float mn = fmaxf(m, tmax);            // key t0 is always valid: mn is finite
    const float alpha = exp2f(m - mn);          // m = -inf on the first tile -> 0
    const float p00 = exp2f(s[0][0] - mn), p01 = exp2f(s[0][1] - mn), p10 = exp2f(s[1][0] - mn), p11 = exp2f(s[1][1] - mn);
    l = l * alpha + (p00 + p01) + (p10 + p11);
    m = mn;
    const uint32_t pa0 = pack2_bf16(p00, p01), pa2 = pack2_bf16(p10, p11);
#pragma unroll
    for (int c = 0; c < 16; c += 2) {
      uint32_t bv[4];
      const int key = (lm & 1) * 8 + lr;
      dec_ldsm_t(bv, vt + key * 256 + (((c + (lm >> 1)) ^ (key & 7)) << 4));
      o[c][0] *= alpha; o[c][1] *= alpha; o[c + 1][0] *= alpha; o[c + 1][1] *= alpha;
      mma_m16n8k16(o[c], pa0, pa2, bv[0], bv[1]);
      mma_m16n8k16(o[c + 1], pa0, pa2, bv[2], bv[3]);
    }
    __syncwarp();                               // the stage may be refilled by the next issue_tile()
    st_done = (st_done == (kDecStages - 1) * kDecTileBytes) ? 0u : st_done + kDecTileBytes;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  l += __shfl_xor_sync(0xffffffffu, l, 1);
  l += __shfl_xor_sync(0xffffffffu, l, 2);
  __syncthreads();                              // every warp is done with its ring: reuse it for the merge
  float* sm_o = reinterpret_cast<float*>(dec_smem);                    // [kDecWarps][8][HD]
  float* sm_m = sm_o + kDecWarps * 8 * HD;                             // [kDecWarps][8]
  float* sm_l = sm_m + kDecWarps * 8;
  if (t == 0) { sm_m[w * 8 + g] = m; sm_l[w * 8 + g] = l; }
#pragma unroll
  for (int j = 0; j < 16; ++j)
    *reinterpret_cast<float2*>(&sm_o[(w * 8 + g) * HD + j * 8 + 2 * t]) = make_float2(o[j][0], o[j][1]);
  __syncthreads();
  const int d = threadIdx.x;   // kDecWarps * 32 == HD
  for (int r = 0; r < G; ++r) {
    float mm = -INFINITY;
#pragma unroll
    for (int ww = 0; ww < kDecWarps; ++ww) mm = fmaxf(mm, sm_m[ww * 8 + r]);
    float num = 0.f, den = 0.f;
#pragma unroll
    for (int ww = 0; ww < kDecWarps; ++ww) {
      const float f = (sm_m[ww * 8 + r] == -INFINITY) ? 0.f : exp2f(sm_m[ww * 8 + r] - mm);
      num += sm_o[(ww * 8 + r) * HD + d] * f;
      den += sm_l[ww * 8 + r] * f;
    }
    // partial record per (b, head, split): [m, l, pad, pad, acc[128]]
    float* rec = part + (((long long)b * kv_heads * G + kvh * G + r) * kDecSplits + sp) * (HD + 4);
    if (d == 0) { rec[0] = mm; rec[1] = den; }
    rec[4 + d] = num;
  }
}

// merge the kDecSplits partials of one (sequence, q head): out = sum_s acc_s * 2^(m_s - m) / sum_s l_s * 2^(m_s - m)
__global__ void __launch_bounds__(128) decode_attn_combine_kernel(const float* __restrict__ part, bf16* __restrict__ out, long long ldo,
                                                                  int q_heads, int n_splits) {
  constexpr int HD = 128;
  const int b = blockIdx.x, h = blockIdx.y, d = threadIdx.x;
  griddep_launch();
  griddep_wait();
  const float* rec = part + (((long long)b * q_heads + h) * kDecSplits) * (HD + 4);
  float mm = -INFINITY;
#pragma unroll
  for (int s = 0; s < n_splits; ++s) mm = fmaxf(mm, rec[s * (HD + 4)]);
  float num = 0.f, den = 0.f;
#pragma unroll
  for (int s = 0; s < n_splits; ++s) {
    const float ms = rec[s * (HD + 4)];
    const float sc = (ms == -INFINITY) ? 0.f : exp2f(ms - mm);
    num += rec[s * (HD + 4) + 4 + d] * sc;
    den += rec[s * (HD + 4) + 1] * sc;
  }
  out[(long long)b * ldo + (long long)h * HD + d] = __float2bfloat16_rn(num / den);
}

// host side of the decode attention: split count = one wave of blocks (2 per SM: 96 KB of shared memory each)
static int decode_attention(const bf16* q, long long ldq, const bf16* kc, const bf16* vc, const int* cache_len, int rows, int cap,
                            int q_heads, int kv_heads, int hd, float scale, bf16* out, long long ldo, float* part, cudaStream_t s) {
  const int G = kv_heads > 0 ? q_heads / kv_heads : 0;
  if (kv_heads <= 0 || q_heads % kv_heads != 0 || G > 8 || hd != 128) {
    set_error("decode attention: %d/%d heads, head_dim %d unsupported (GQA group <= 8, head_dim 128)", q_heads, kv_heads, hd);
    return FO1_ERR_UNSUPPORTED;
  }
  if (rows == 0) return FO1_OK;
  static bool attr_set = false;
  if (!attr_set) { FO1_CUDA(cudaFuncSetAttribute(decode_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kDecSmemBytes)); attr_set = true; }
  const int slots = 2 * device_sm_count();
  const int n_splits = std::max(1, std::min(kDecSplits, slots / std::max(1, rows * kv_heads)));
  dim3 grid(rows, kv_heads, n_splits);
  ProfScope prof("decode_attn", 0.0, 0.0, s);
  launch_k(decode_attn_kernel, grid, dim3(kDecWarps * 32), kDecSmemBytes, s, q, ldq, kc, vc, cache_len, cap, kv_heads, G, part, scale);
  FO1_LAUNCH_CHECK();
  launch_k(decode_attn_combine_kernel, dim3(rows, q_heads), dim3(128), 0, s, (const float*)part, out, ldo, q_heads, n_splits);
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}

// greedy token: lowest index among the maxima of a fp32 logits row
__global__ void __launch_bounds__(1024) argmax_kernel(const float* __restrict__ logits, int V, int* __restrict__ out) {
  griddep_launch();
  griddep_wait();
  const float* row = logits + (long long)blockIdx.x * V;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = threadIdx.x; i < V; i += blockDim.x) {
    const float v = row[i];
    if (v > best || (v == best && i < bi)) { best = v; bi = i; }
  }
  __shared__ float sv[32];
  __shared__ int si[32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
  }
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = best; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  if (threadIdx.x < 32) {
    best = sv[threadIdx.x]; bi = si[threadIdx.x];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    if (threadIdx.x == 0) out[blockIdx.x] = bi;
  }
}

struct DecodeState {
  int* cache_len;  // [B] K/V entries in the cache
  int* pos3;       // [3][B] M-RoPE position of the next input token (all axes equal after the prompt, :1848-1860)
  int* cur_tok;    // [B] token to feed next
  int* new_tok;    // [B] argmax output
  int* finished;   // [B]
  int* n_active;   // [1] sequences still running
  int* step;       // [1] index of the next output column
  int* stop_ids;   // [n_stop]
};

// after the prefill: lengths, positions, first token
__global__ void decode_init_kernel(DecodeState st, const int* __restrict__ seq_lens, const int* __restrict__ deltas, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b == 0) { *st.step = 0; *st.n_active = B; }
  if (b >= B) return;
  st.cache_len[b] = seq_lens[b];
  const int p = seq_lens[b] + deltas[b];
  st.pos3[b] = p; st.pos3[B + b] = p; st.pos3[2 * B + b] = p;
  st.finished[b] = 0;
}
// record the sampled token, test the stop ids, advance the loop state.  ONE block; the output column is the
// device-resident step counter, so the launch is identical every iteration (CUDA-graph replayable).
__global__ void __launch_bounds__(1024) decode_update_kernel(DecodeState st, int n_stop, int pad_id, int max_new,
                                                             int* __restrict__ out_tokens, int* __restrict__ out_lens, int B,
                                                             int advance_cache) {
  griddep_launch();
  griddep_wait();
  const int step = *st.step;
  __syncthreads();
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const int tok = st.new_tok[b];
    if (step < max_new) {
      if (!st.finished[b]) {
        out_tokens[(long long)b * max_new + step] = tok;
        out_lens[b] = step + 1;
        bool stop = false;
        for (int i = 0; i < n_stop; ++i) stop |= (tok == st.stop_ids[i]);
        if (stop) { st.finished[b] = 1; atomicSub(st.n_active, 1); }
      } else {
        out_tokens[(long long)b * max_new + step] = pad_id;
      }
    }
    st.cur_tok[b] = tok;
    if (advance_cache) {
      st.cache_len[b] += 1;
      st.pos3[b] += 1; st.pos3[B + b] += 1; st.pos3[2 * B + b] += 1;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) *st.step = step + 1;
}
__global__ void fill_int_kernel(int* p, int v, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) p[i] = v;
}

// ------------------------------------------------------------------------------------------ host
struct LlmState {
  int* ints = nullptr;   // one allocation for the DecodeState arrays
  int cap_b = 0, cap_stop = 0;
  int* h_flag = nullptr; // pinned
};

static int llm_resolve(Model* m) {
  const fo1_model_config& c = m->cfg;
  WeightGetter g{m, ""};
  LlmW& w = m->llm;
  const int64_t H = c.llm_hidden, V = c.llm_vocab, QD = (int64_t)c.llm_heads * c.llm_head_dim, KD = (int64_t)c.llm_kv_heads * c.llm_head_dim;
  const int64_t Ip = (c.llm_inter + 31) / 32 * 32;
  w.embed = g.bf("llm.embed", {V, H});
  w.norm = g.bf("llm.norm.w", {H});
  w.lm_head = g.bf("llm.lm_head", {V, H});
  w.layer.resize(c.llm_layers);
  for (int i = 0; i < c.llm_layers; ++i) {
    const std::string p = "llm.l" + std::to_string(i) + ".";
    LlmLayerW& L = w.layer[i];
    L.ln1 = g.bf(p + "ln1.w", {H});
    L.qkv_w = g.bf(p + "qkv.w", {QD + 2 * KD, H});
    L.qkv_b = g.bf(p + "qkv.b", {QD + 2 * KD});
    L.o_w = g.bf(p + "o.w", {H, QD});
    L.ln2 = g.bf(p + "ln2.w", {H});
    L.gateup_w = g.bf(p + "gateup.w", {2 * Ip, H});
    L.down_w = g.bf(p + "down.w", {H, Ip});
  }
  if (!g.err.empty()) { set_error("LLM weights: %s", g.err.c_str()); return FO1_ERR_NOT_FOUND; }
  w.ok = true;
  // optional decode copies (weights.py::prepare_llm): W diag(g) for the two normed projections and the LM head, gate / up in the
  // decode kernel's 8 + 8 row interleave.  All present -> the persistent decode kernel is used.
  w.mega_ok = m->find("llm.head_dec") != nullptr;
  for (int i = 0; i < c.llm_layers && w.mega_ok; ++i) {
    const std::string p = "llm.l" + std::to_string(i) + ".";
    w.mega_ok = m->find(p + "qkv_dec.w") != nullptr && m->find(p + "gu_dec.w") != nullptr;
  }
  if (w.mega_ok) {
    WeightGetter g2{m, ""};
    w.head_dec = g2.bf("llm.head_dec", {V, H});
    std::vector<MegaLayer> ml(c.llm_layers);
    for (int i = 0; i < c.llm_layers; ++i) {
      const std::string p = "llm.l" + std::to_string(i) + ".";
      LlmLayerW& L = w.layer[i];
      L.qkv_dec = g2.bf(p + "qkv_dec.w", {QD + 2 * KD, H});
      L.gu_dec = g2.bf(p + "gu_dec.w", {2 * (int64_t)c.llm_inter, H});
      ml[i].qkv_w = L.qkv_dec; ml[i].qkv_b = L.qkv_b; ml[i].o_w = L.o_w; ml[i].gu_w = L.gu_dec; ml[i].down_w = L.down_w;
    }
    if (!g2.err.empty()) { set_error("LLM decode weights: %s", g2.err.c_str()); return FO1_ERR_NOT_FOUND; }
    if (c.llm_inter != Ip) w.mega_ok = false;      // the decode kernel reads down_w with K = intermediate size (no padding)
    if (w.mega_ok) {
      if (w.mega_layers) cudaFree(w.mega_layers);
      FO1_CUDA(cudaMalloc(&w.mega_layers, ml.size() * sizeof(MegaLayer)));
      FO1_CUDA(cudaMemcpy(w.mega_layers, ml.data(), ml.size() * sizeof(MegaLayer), cudaMemcpyHostToDevice));
    }
  }
  return FO1_OK;
}
int llm_finalize(Model* m) { return m->cfg.llm_layers > 0 ? llm_resolve(m) : FO1_OK; }

void llm_destroy_state(Model* m) {
  if (m->llm.mega_layers) { cudaFree(m->llm.mega_layers); m->llm.mega_layers = nullptr; }
  LlmState* s = static_cast<LlmState*>(m->llm_state);
  if (!s) return;
  if (s->ints) cudaFree(s->ints);
  if (s->h_flag) cudaFreeHost(s->h_flag);
  delete s;
  m->llm_state = nullptr;
}

static int ensure_kv(Model* m, int B, int cap) {
  const fo1_model_config& c = m->cfg;
  const size_t per = (size_t)c.llm_layers * B * cap * c.llm_kv_heads * c.llm_head_dim * sizeof(bf16);
  if (2 * per > m->kv_bytes) {
    FO1_CUDA(cudaDeviceSynchronize());
    if (m->kv_cache) FO1_CUDA(cudaFree(m->kv_cache));
    m->kv_cache = nullptr; m->kv_bytes = 0;
    FO1_CUDA(cudaMalloc(&m->kv_cache, 2 * per));
    m->kv_bytes = 2 * per;
  }
  m->kv_batch = B; m->kv_cap = cap;
  return FO1_OK;
}

static int ensure_state(Model* m, int B, int n_stop, DecodeState* st) {
  LlmState* s = static_cast<LlmState*>(m->llm_state);
  if (!s) { s = new LlmState(); m->llm_state = s; }
  if (B > s->cap_b || n_stop > s->cap_stop) {
    FO1_CUDA(cudaDeviceSynchronize());
    if (s->ints) FO1_CUDA(cudaFree(s->ints));
    s->cap_b = std::max(B, s->cap_b); s->cap_stop = std::max(n_stop, std::max(s->cap_stop, 8));
    FO1_CUDA(cudaMalloc(reinterpret_cast<void**>(&s->ints), ((size_t)9 * s->cap_b + s->cap_stop + 64) * sizeof(int)));
  }
  if (!s->h_flag) FO1_CUDA(cudaMallocHost(reinterpret_cast<void**>(&s->h_flag), 64));
  int* p = s->ints;
  const int cb = s->cap_b;
  st->cache_len = p; p += cb;
  st->pos3 = p; p += 3 * cb;
  st->cur_tok = p; p += cb;
  st->new_tok = p; p += cb;
  st->finished = p; p += cb;
  st->n_active = p; p += 16;
  st->step = p; p += 16;
  st->stop_ids = p;
  return FO1_OK;
}

// one decoder layer over `rows` packed rows.  x_in -> x_out (x_mid scratch).  prefill: varlen causal attention
// + cache fill; decode: cache append + single-query attention.
struct LayerBuf { bf16 *xn, *qkv, *att, *x_mid, *h; float* dec_part; int* rowseg = nullptr; double attn_flops = 0.0; const int* tiles = nullptr; int n_tiles = 0; };

static int llm_layer(Model* m, int li, const bf16* x_in, bf16* x_out, const LayerBuf& B_, int rows, const float* cs, bool prefill,
                     const int* d_cu, int n_seqs, int max_len, const int* d_row_seq, const int* d_row_t, const DecodeState* st,
                     cudaStream_t s, bool dry) {
  const fo1_model_config& c = m->cfg;
  const LlmLayerW& L = m->llm.layer[li];
  const int H = c.llm_hidden, hd = c.llm_head_dim, QD = c.llm_heads * hd, KD = c.llm_kv_heads * hd, ldq = QD + 2 * KD;
  const int Ip = (c.llm_inter + 31) / 32 * 32;
  const size_t layer_stride = (size_t)m->kv_batch * m->kv_cap * KD;
  bf16* kc = static_cast<bf16*>(m->kv_cache) + (size_t)li * layer_stride;
  bf16* vc = static_cast<bf16*>(m->kv_cache) + ((size_t)c.llm_layers + li) * layer_stride;
  FO1_RUN(rmsnorm(x_in, H, L.ln1, B_.xn, H, rows, H, c.rms_eps, s));
  FO1_RUN(linear(B_.xn, H, L.qkv_w, H, B_.qkv, ldq, FO1_BF16, rows, ldq, H, L.qkv_b, FO1_BF16, FO1_EPI_NONE, nullptr, 0, 0, s));
  if (prefill) {
    FO1_RUN(rope_apply(B_.qkv, ldq, cs, rows, c.llm_heads + c.llm_kv_heads, hd, s));   // q|k heads are contiguous in the packed row
    if (!dry) {
      kv_store_kernel<<<rows, 128, 0, s>>>(B_.qkv, ldq, QD, KD, d_row_seq, d_row_t, kc, vc, m->kv_cap);
      FO1_LAUNCH_CHECK();
    }
    AttnArgs a;
    a.q = B_.qkv; a.k = B_.qkv + QD; a.v = B_.qkv + QD + KD; a.o = B_.att;
    a.ldq = a.ldk = a.ldv = ldq; a.ldo = QD;
    a.cu_seqlens = d_cu; a.n_seqs = n_seqs; a.max_seqlen = max_len; a.total_rows = rows; a.rowseg = B_.rowseg; a.flops = B_.attn_flops; a.tiles = B_.tiles; a.n_tiles = B_.n_tiles;
    a.q_heads = c.llm_heads; a.kv_heads = c.llm_kv_heads; a.head_dim = hd;
    a.scale = 1.0f / sqrtf((float)hd); a.causal = 1;
    FO1_RUN(attention_varlen(a, s));
  } else if (!dry) {
    FO1_RUN(rope_kv_append(B_.qkv, ldq, cs, rows, c.llm_heads, c.llm_kv_heads, hd, st->cache_len, kc, vc, m->kv_cap, s));
    FO1_RUN(decode_attention(B_.qkv, ldq, kc, vc, st->cache_len, rows, m->kv_cap, c.llm_heads, c.llm_kv_heads, hd,
                             1.0f / sqrtf((float)hd), B_.att, QD, B_.dec_part, s));
  }
  FO1_RUN(linear(B_.att, QD, L.o_w, QD, B_.x_mid, H, FO1_BF16, rows, H, QD, nullptr, 0, FO1_EPI_NONE, x_in, H, 0, s));
  FO1_RUN(rmsnorm(B_.x_mid, H, L.ln2, B_.xn, H, rows, H, c.rms_eps, s));
  FO1_RUN(linear(B_.xn, H, L.gateup_w, H, B_.h, Ip, FO1_BF16, rows, 2 * Ip, H, nullptr, 0, FO1_EPI_SILU, nullptr, 0, 1, s));
  FO1_RUN(linear(B_.h, Ip, L.down_w, Ip, x_out, H, FO1_BF16, rows, H, Ip, nullptr, 0, FO1_EPI_NONE, B_.x_mid, H, 0, s));
  return FO1_OK;
}

static int llm_generate_impl(Model* m, fo1_generate_desc* d, cudaStream_t s, bool dry, const DecodeState& st) {
  const fo1_model_config& c = m->cfg;
  Arena& A = m->arena;
  const int B = d->n_seqs, H = c.llm_hidden, hd = c.llm_head_dim, V = c.llm_vocab;
  const int QD = c.llm_heads * hd, KD = c.llm_kv_heads * hd, ldq = QD + 2 * KD;
  const int Ip = (c.llm_inter + 31) / 32 * 32;
  long long T = 0;
  int max_len = 0;
  for (int b = 0; b < B; ++b) { T += d->seq_lens[b]; max_len = std::max(max_len, d->seq_lens[b]); }
  const int R = (int)std::max<long long>(T, B);

  LayerBuf buf;
  bf16* xa = A.alloc<bf16>((size_t)R * H);
  bf16* xb = A.alloc<bf16>((size_t)R * H);
  buf.xn = A.alloc<bf16>((size_t)R * H);
  buf.qkv = A.alloc<bf16>((size_t)R * ldq);
  buf.att = A.alloc<bf16>((size_t)R * QD);
  buf.x_mid = A.alloc<bf16>((size_t)R * H);
  buf.h = A.alloc<bf16>((size_t)R * Ip);
  float* cs_pre = A.alloc<float>((size_t)R * hd);
  float* cs_dec = A.alloc<float>((size_t)B * hd);
  buf.dec_part = A.alloc<float>((size_t)B * c.llm_heads * kDecSplits * (128 + 4));
  buf.rowseg = A.alloc<int>((size_t)R * 2);
  for (int b = 0; b < B; ++b) buf.attn_flops += 2.0 * (double)d->seq_lens[b] * d->seq_lens[b] * QD;   // causal: half of 4 L^2 d
  bf16* last = A.alloc<bf16>((size_t)B * H);
  bf16* lastn = A.alloc<bf16>((size_t)B * H);
  float* logits = A.alloc<float>((size_t)B * V);
  bf16* alln = d->all_logits ? A.alloc<bf16>((size_t)T * H) : nullptr;
  int* d_lens = A.alloc<int>(B);
  int* d_deltas = A.alloc<int>(B);
  // persistent decode kernel (decode_mega.cu): per-CTA slots + the grid barrier
  // measured with warm clocks, alternating the two paths (scripts/mega_prof.py, profiles/README.md round 2): the persistent kernel
  // beats the per-kernel graph at every batch it supports (1..32 sequences: -8 % .. -19 % per step).  FO1_NO_MEGA disables the
  // kernel.
  const int mega_grid = (m->llm.mega_ok && B <= 32 && getenv("FO1_NO_MEGA") == nullptr) ? decode_mega_grid() : 0;
  float* mg_ssq = A.alloc<float>((size_t)2 * std::max(mega_grid, 1) * 32);
  float* mg_amax_v = A.alloc<float>((size_t)std::max(mega_grid, 1) * 32);
  int* mg_amax_i = A.alloc<int>((size_t)std::max(mega_grid, 1) * 32);
  int* mg_sync = A.alloc<int>((size_t)B * c.llm_kv_heads + 8);      // [0]: grid barrier counter, [8..]: attention arrival counters

  // ---- integer tables of the packed batch ----
  const int *d_cu = nullptr, *d_row_seq = nullptr, *d_row_t = nullptr, *d_last = nullptr;
  if (!dry) {
    std::vector<int> cu(1, 0), row_seq, row_t, lastrow;
    std::string key = "llm";
    for (int b = 0; b < B; ++b) {
      for (int t = 0; t < d->seq_lens[b]; ++t) { row_seq.push_back(b); row_t.push_back(t); }
      cu.push_back(cu.back() + d->seq_lens[b]);
      lastrow.push_back(cu.back() - 1);
      key += ":" + std::to_string(d->seq_lens[b]);
    }
    FO1_TRY(cached_ints(m, key + ":cu", cu, &d_cu, s));
    FO1_TRY(cached_ints(m, key + ":rs", row_seq, &d_row_seq, s));
    FO1_TRY(cached_ints(m, key + ":rt", row_t, &d_row_t, s));
    FO1_TRY(cached_ints(m, key + ":last", lastrow, &d_last, s));
    std::vector<int> tiles;
    attention_tile_table(cu, tiles);        // query tiles restart at every prompt
    FO1_TRY(cached_ints(m, key + ":til", tiles, &buf.tiles, s));
    buf.n_tiles = (int)tiles.size() / 2;
    FO1_CUDA(cudaMemcpyAsync(d_lens, d->seq_lens, B * sizeof(int), cudaMemcpyHostToDevice, s));
    if (d->rope_deltas_device != nullptr) FO1_CUDA(cudaMemcpyAsync(d_deltas, d->rope_deltas_device, B * sizeof(int), cudaMemcpyDeviceToDevice, s));
    else FO1_CUDA(cudaMemcpyAsync(d_deltas, d->rope_deltas, B * sizeof(int), cudaMemcpyHostToDevice, s));
    if (d->n_stop_ids > 0) FO1_CUDA(cudaMemcpyAsync(st.stop_ids, d->stop_ids, d->n_stop_ids * sizeof(int), cudaMemcpyHostToDevice, s));
  }

  // ---- prefill ----
  FO1_RUN(attention_rowseg(d_cu, B, (int)T, buf.rowseg, s));
  const bf16* x = static_cast<const bf16*>(d->inputs_embeds);
  FO1_RUN(mrope_table(d->position_ids, cs_pre, (int)T, hd, c.mrope_section[0], c.mrope_section[1], c.mrope_section[2], c.rope_theta, s));
  for (int li = 0; li < c.llm_layers; ++li) {
    bf16* xo = (li & 1) ? xb : xa;
    FO1_TRY(llm_layer(m, li, x, xo, buf, (int)T, cs_pre, true, d_cu, B, max_len, d_row_seq, d_row_t, nullptr, s, dry));
    x = xo;
  }
  if (d->all_logits) {
    FO1_RUN(rmsnorm(x, H, m->llm.norm, alln, H, (int)T, H, c.rms_eps, s));
    FO1_RUN(linear(alln, H, m->llm.lm_head, H, d->all_logits, V, FO1_F32, (int)T, V, H, nullptr, 0, FO1_EPI_NONE, nullptr, 0, 0, s));
  }
  FO1_RUN(gather_rows_bf16(x, H, d_last, last, H, B, H, s));
  FO1_RUN(rmsnorm(last, H, m->llm.norm, lastn, H, B, H, c.rms_eps, s));
  {
    SplitKScope sk(true);       // M = number of sequences: weight streaming
    FO1_RUN(linear(lastn, H, m->llm.lm_head, H, logits, V, FO1_F32, B, V, H, nullptr, 0, FO1_EPI_NONE, nullptr, 0, 0, s));
  }
  if (dry) return FO1_OK;
  if (d->prefill_logits) FO1_CUDA(cudaMemcpyAsync(d->prefill_logits, logits, (size_t)B * V * sizeof(float), cudaMemcpyDeviceToDevice, s));
  decode_init_kernel<<<ceil_div(B, 128), 128, 0, s>>>(st, d_lens, d_deltas, B);
  FO1_LAUNCH_CHECK();
  if (d->max_new_tokens <= 0) return FO1_OK;
  argmax_kernel<<<B, 1024, 0, s>>>(logits, V, st.new_tok);
  FO1_LAUNCH_CHECK();
  const int upd_threads = std::min(1024, std::max(32, (B + 31) / 32 * 32));
  decode_update_kernel<<<1, upd_threads, 0, s>>>(st, d->n_stop_ids, d->pad_id, d->max_new_tokens, d->out_tokens, d->out_lens, B, 0);
  FO1_LAUNCH_CHECK();

  // ---- greedy decode: every step is the SAME launch sequence reading its state from device memory; the first
  // step runs eagerly (warms every kernel), the second is captured into a CUDA graph that is replayed afterwards ----
  LlmState* ls = static_cast<LlmState*>(m->llm_state);
  // programmatic dependent launch: each kernel of the step starts (prologue, weight prefetch) while its predecessor drains
  auto enqueue_step = [&]() -> int {
    PdlScope pdl(true);
    SplitKScope sk(true);       // M = number of sequences in every GEMM of a decode step
    launch_k(embed_tokens_kernel, dim3(B), dim3(256), 0, s, st.cur_tok, m->llm.embed, xa, H);
    FO1_LAUNCH_CHECK();
    FO1_TRY(mrope_table(st.pos3, cs_dec, B, hd, c.mrope_section[0], c.mrope_section[1], c.mrope_section[2], c.rope_theta, s));
    const bf16* xin = xa;
    for (int li = 0; li < c.llm_layers; ++li) {
      bf16* xo = (li & 1) ? xa : xb;
      FO1_TRY(llm_layer(m, li, xin, xo, buf, B, cs_dec, false, nullptr, B, 0, nullptr, nullptr, &st, s, false));
      xin = xo;
    }
    FO1_TRY(rmsnorm(xin, H, m->llm.norm, lastn, H, B, H, c.rms_eps, s));
    FO1_TRY(linear(lastn, H, m->llm.lm_head, H, logits, V, FO1_F32, B, V, H, nullptr, 0, FO1_EPI_NONE, nullptr, 0, 0, s));
    launch_k(argmax_kernel, dim3(B), dim3(1024), 0, s, logits, V, st.new_tok);
    FO1_LAUNCH_CHECK();
    launch_k(decode_update_kernel, dim3(1), dim3(upd_threads), 0, s, st, d->n_stop_ids, d->pad_id, d->max_new_tokens, d->out_tokens, d->out_lens, B, 1);
    FO1_LAUNCH_CHECK();
    return FO1_OK;
  };
  if (mega_grid > 0 && d->max_new_tokens > 1) {
    // ---- the whole greedy loop as ONE cooperative launch ----
    MegaArgs a;
    memset(&a, 0, sizeof(a));
    a.B = B; a.layers = c.llm_layers; a.H = H; a.QD = QD; a.KD = KD; a.hd = hd; a.q_heads = c.llm_heads; a.kv_heads = c.llm_kv_heads;
    a.I = c.llm_inter; a.V = V; a.eps = c.rms_eps; a.theta = c.rope_theta; a.sec_t = c.mrope_section[0]; a.sec_h = c.mrope_section[1];
    a.layer = static_cast<const MegaLayer*>(m->llm.mega_layers);
    a.head_w = m->llm.head_dec; a.embed = m->llm.embed;
    a.kv_layer_stride = (long long)m->kv_batch * m->kv_cap * KD;
    a.kc = static_cast<bf16*>(m->kv_cache);
    a.vc = static_cast<bf16*>(m->kv_cache) + (size_t)c.llm_layers * a.kv_layer_stride;
    a.cap = m->kv_cap;
    a.x = xa; a.x_mid = buf.x_mid; a.qkv = buf.qkv; a.att = buf.att; a.h = buf.h;
    a.ssq = mg_ssq; a.cs = cs_dec; a.att_part = buf.dec_part; a.att_count = mg_sync + 8;
    a.amax_val = mg_amax_v; a.amax_idx = mg_amax_i;
    a.cache_len = st.cache_len; a.pos3 = st.pos3; a.cur_tok = st.cur_tok; a.finished = st.finished; a.n_active = st.n_active; a.step = st.step;
    a.stop_ids = st.stop_ids; a.n_stop = d->n_stop_ids; a.pad_id = d->pad_id; a.max_new = d->max_new_tokens;
    a.out_tokens = d->out_tokens; a.out_lens = d->out_lens;
    a.n_steps = d->max_new_tokens - 1;
    a.bar = reinterpret_cast<unsigned*>(mg_sync);
    const int pairs = B * c.llm_kv_heads;
    a.n_splits = std::max(1, std::min(kMgMaxSplits, mega_grid / std::max(1, pairs)));
    FO1_CUDA(cudaMemsetAsync(mg_sync, 0, ((size_t)pairs + 8) * sizeof(int), s));
    unsigned long long* d_prof = nullptr;
    const int prof_slots = 5 * c.llm_layers + 3 + 8;     // + 8 sub-stamps of one attention item (CTA 0, layer 1)
    if (getenv("FO1_MEGA_PROF") != nullptr) {       // diagnostic: where a decode iteration spends its time (stderr)
      FO1_CUDA(cudaMalloc(reinterpret_cast<void**>(&d_prof), (size_t)mega_grid * prof_slots * 2 * sizeof(unsigned long long)));
      FO1_CUDA(cudaMemsetAsync(d_prof, 0, (size_t)mega_grid * prof_slots * 2 * sizeof(unsigned long long), s));
      a.prof = d_prof; a.prof_slots = prof_slots;
    }
    FO1_TRY(decode_mega_run(a, s));
    m->last_decode_path = 1;
    if (d_prof != nullptr) {
      std::vector<unsigned long long> h((size_t)mega_grid * prof_slots * 2);
      FO1_CUDA(cudaStreamSynchronize(s));
      FO1_CUDA(cudaMemcpy(h.data(), d_prof, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
      cudaFree(d_prof);
      // per slot: the last CTA to enter the barrier ends the phase; release = when CTA 0 leaves.  work = last_enter - previous release,
      // skew = last_enter - first_enter, barrier = release - last_enter
      const char* names[5] = {"qkv", "attn", "oproj", "gateup", "down"};
      double tot[5][3] = {{0}}, misc = 0;
      unsigned long long prev_release = 0;
      for (int sl = 0; sl < prof_slots - 8; ++sl) {
        unsigned long long first = ~0ull, last = 0, rel = 0;
        for (int cta = 0; cta < mega_grid; ++cta) {
          const unsigned long long e = h[((size_t)cta * prof_slots + sl) * 2], l = h[((size_t)cta * prof_slots + sl) * 2 + 1];
          if (e < first) first = e;
          if (e > last) last = e;
          if (l > rel) rel = l;
        }
        if (sl >= 1 && sl <= 5 * c.llm_layers) {
          const int ph = (sl - 1) % 5;
          tot[ph][0] += (double)(last - prev_release); tot[ph][1] += (double)(last - first); tot[ph][2] += (double)(rel - last);
        } else if (sl > 0) misc += (double)(rel - prev_release);
        prev_release = rel;
      }
      fprintf(stderr, "[decode_mega profile, first iteration, B=%d, %d CTAs] per layer (us): ", B, mega_grid);
      for (int ph = 0; ph < 5; ++ph)
        fprintf(stderr, "%s work %.1f (skew %.1f) barrier %.1f | ", names[ph], tot[ph][0] / c.llm_layers / 1e3, tot[ph][1] / c.llm_layers / 1e3,
                tot[ph][2] / c.llm_layers / 1e3);
      fprintf(stderr, "head+update %.1f us\n", misc / 1e3);
      {   // distribution over CTAs of the time spent in layer 1's attention phase (slot 7: enter of the barrier after it; slot 6: leave before it)
        std::vector<std::pair<double, int>> dur;
        for (int cta = 0; cta < mega_grid; ++cta)
          dur.push_back({(double)(h[((size_t)cta * prof_slots + 7) * 2] - h[((size_t)cta * prof_slots + 6) * 2 + 1]) / 1e3, cta});
        std::sort(dur.begin(), dur.end());
        fprintf(stderr, "[decode_mega profile] attention phase per CTA (us): min %.1f p25 %.1f median %.1f p75 %.1f max %.1f; slowest CTAs:", dur[0].first,
                dur[mega_grid / 4].first, dur[mega_grid / 2].first, dur[3 * mega_grid / 4].first, dur.back().first);
        for (int k = 0; k < 6; ++k) fprintf(stderr, " %d(%.1f)", dur[mega_grid - 1 - k].second, dur[mega_grid - 1 - k].first);
        fprintf(stderr, "\n");
      }
      fprintf(stderr, "[decode_mega profile] attention item of CTA 0, layer 1 (us since its start): ");
      const unsigned long long a0 = h[((size_t)0 * prof_slots + prof_slots - 8) * 2];
      const char* an[8] = {"start", "append+fence", "q rotated", "tiles done", "warps synced", "partials written", "fence+sync", "combined"};
      for (int k = 0; k < 8; ++k) fprintf(stderr, "%s %.1f | ", an[k], (double)(h[((size_t)0 * prof_slots + prof_slots - 8 + k) * 2] - a0) / 1e3);
      fprintf(stderr, "\n");
    }
    d->steps_run = d->max_new_tokens - 1;
    return FO1_OK;
  }
  cudaGraphExec_t gexec = nullptr;
  m->last_decode_path = 0;
  const bool want_graph = !g_prof_on && d->max_new_tokens > 3;
  d->steps_run = 0;
  int rc = FO1_OK;
  for (int step = 1; step < d->max_new_tokens; ++step) {
    if (gexec != nullptr) {
      if (cudaGraphLaunch(gexec, s) != cudaSuccess) { set_error("cudaGraphLaunch failed: %s", cudaGetErrorString(cudaGetLastError())); rc = FO1_ERR_CUDA; break; }
      count_launch((uint64_t)c.llm_layers * 9 + 6);
    } else if (want_graph && step == 2) {
      cudaGraph_t graph = nullptr;
      if (cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
        const int erc = enqueue_step();
        const cudaError_t ce = cudaStreamEndCapture(s, &graph);
        if (erc == FO1_OK && ce == cudaSuccess && graph != nullptr && cudaGraphInstantiate(&gexec, graph, 0) == cudaSuccess) {
          cudaGraphDestroy(graph);
          if (cudaGraphLaunch(gexec, s) != cudaSuccess) { set_error("cudaGraphLaunch failed"); rc = FO1_ERR_CUDA; break; }
        } else {  // capture unavailable: fall back to eager launches (still the same kernels)
          if (graph) cudaGraphDestroy(graph);
          cudaGetLastError();
          gexec = nullptr;
          if ((rc = enqueue_step()) != FO1_OK) break;
        }
      } else {
        cudaGetLastError();
        if ((rc = enqueue_step()) != FO1_OK) break;
      }
    } else {
      if ((rc = enqueue_step()) != FO1_OK) break;
    }
    d->steps_run = step;
    if (d->early_exit_interval > 0 && step % d->early_exit_interval == 0) {
      if (cudaMemcpyAsync(ls->h_flag, st.n_active, sizeof(int), cudaMemcpyDeviceToHost, s) != cudaSuccess || cudaStreamSynchronize(s) != cudaSuccess) {
        set_error("early-exit poll failed"); rc = FO1_ERR_CUDA; break;
      }
      if (*ls->h_flag <= 0) break;  // every sequence has emitted a stop id; the tail is already pad_id
    }
  }
  if (gexec != nullptr) {
    cudaStreamSynchronize(s);   // the exec must outlive its in-flight launches
    cudaGraphExecDestroy(gexec);
  }
  return rc;
}

int llm_generate(Model* m, fo1_generate_desc* d, cudaStream_t s) {
  FO1_CHECK_ARG(m->llm.ok, "fo1_llm_generate: model not finalized (LLM weights unresolved)");
  const fo1_model_config& c = m->cfg;
  FO1_CHECK_ARG(d->n_seqs > 0 && d->seq_lens && d->inputs_embeds && d->position_ids && (d->rope_deltas || d->rope_deltas_device),
                "fo1_llm_generate: null argument");
  FO1_CHECK_ARG(d->max_new_tokens == 0 || (d->out_tokens && d->out_lens), "fo1_llm_generate: null outputs");
  FO1_CHECK_ARG(c.llm_head_dim == 128, "fo1_llm_generate: head_dim %d unsupported (128)", c.llm_head_dim);
  int max_len = 0;
  for (int b = 0; b < d->n_seqs; ++b) {
    FO1_CHECK_ARG(d->seq_lens[b] > 0, "fo1_llm_generate: sequence %d is empty", b);
    max_len = std::max(max_len, d->seq_lens[b]);
  }
  DecodeState st;
  FO1_TRY(ensure_state(m, d->n_seqs, d->n_stop_ids, &st));
  FO1_TRY(ensure_kv(m, d->n_seqs, max_len + std::max(d->max_new_tokens, 1)));
  FO1_TRY(int_cache_trim(m));
  m->arena.reset(true);
  FO1_TRY(llm_generate_impl(m, d, s, true, st));
  FO1_TRY(arena_ensure(m, m->arena.peak));
  m->arena.reset(false);
  if (d->max_new_tokens > 0) {  // out_tokens pre-filled with pad so an early exit leaves a clean tail
    const long long n = (long long)d->n_seqs * d->max_new_tokens;
    fill_int_kernel<<<(int)std::min<long long>((n + 255) / 256, 1024), 256, 0, s>>>(d->out_tokens, d->pad_id, n);
    FO1_LAUNCH_CHECK();
    FO1_CUDA(cudaMemsetAsync(d->out_lens, 0, d->n_seqs * sizeof(int), s));
  }
  return llm_generate_impl(m, d, s, false, st);
}

// -------------------------------------------------------------------------------- splice plan (host, integer)
static int splice_plan(const int64_t* ids, int n_ids, const int32_t* grid_hw, int n_images, int n_regions, const fo1_splice_cfg& cf,
                       std::vector<int64_t>& new_ids, std::vector<int>& kind, std::vector<int>& index, std::vector<int>& pos,
                       int* rope_delta) {
  // ---- omchat_qwen2_5_vl.py:318-368: walk the ids, expand image placeholders, keep one slot per region ----
  int cur_img = 0, cur_reg = 0, img_row = 0;
  const int unit = cf.merge * cf.merge;
  for (int i = 0; i < n_ids; ++i) {
    const int64_t t = ids[i];
    if (t == cf.image_placeholder) {
      if (cur_img >= n_images) { set_error("fo1_splice_plan: more image placeholders than images (%d)", n_images); return FO1_ERR_INVALID_ARG; }
      const int n = grid_hw[2 * cur_img] * grid_hw[2 * cur_img + 1] / unit;
      for (int k = 0; k < n; ++k) { new_ids.push_back(cf.image_token_id); kind.push_back(1); index.push_back(img_row + k); }
      img_row += n;
      ++cur_img;
    } else if (t == cf.region_placeholder) {
      if (cur_reg >= n_regions) { set_error("fo1_splice_plan: more region placeholders than region features (%d)", n_regions); return FO1_ERR_INVALID_ARG; }
      new_ids.push_back(cf.region_placeholder); kind.push_back(2); index.push_back(cur_reg++);
    } else {
      new_ids.push_back(t); kind.push_back(0); index.push_back((int)t);
    }
  }
  // ---- get_rope_index (modeling_qwen2_5_vl.py:1625-1699) on the spliced ids, attention mask all ones ----
  const int L = (int)new_ids.size();
  pos.assign((size_t)3 * L, 0);
  int image_nums = 0;
  for (int i = 0; i + 1 < L; ++i)
    if (new_ids[i] == cf.vision_start_token_id && new_ids[i + 1] == cf.image_token_id) ++image_nums;
  // (a vision_start in the last position indexes out of range in the reference; treated as "no image" here)
  int st = 0, image_index = 0;
  long long next_base = 0;   // llm_pos_ids_list[-1].max() + 1
  bool have_any = false;
  auto emit_text = [&](int from, int len, long long base) {
    for (int k = 0; k < len; ++k)
      for (int a = 0; a < 3; ++a) pos[(size_t)a * L + from + k] = (int)(base + k);
  };
  for (int it = 0; it < image_nums; ++it) {
    int ed = -1;
    for (int i = st; i < L; ++i) if (new_ids[i] == cf.image_token_id) { ed = i; break; }
    if (ed < 0 || image_index >= n_images) { set_error("fo1_splice_plan: image token bookkeeping mismatch"); return FO1_ERR_INVALID_ARG; }
    const int lh = grid_hw[2 * image_index] / cf.merge, lw = grid_hw[2 * image_index + 1] / cf.merge;
    ++image_index;
    const int text_len = ed - st;
    const long long st_idx = have_any ? next_base : 0;
    emit_text(st, text_len, st_idx);
    const long long vb = st_idx + text_len;
    for (int y = 0; y < lh; ++y)
      for (int x = 0; x < lw; ++x) {
        const size_t p = (size_t)ed + (size_t)y * lw + x;
        if (p >= (size_t)L) { set_error("fo1_splice_plan: image tokens overrun the sequence"); return FO1_ERR_INVALID_ARG; }
        pos[p] = (int)vb;                     // t index = 0 for an image
        pos[(size_t)L + p] = (int)(vb + y);
        pos[(size_t)2 * L + p] = (int)(vb + x);
      }
    long long mx = vb + std::max(lh, lw) - 1;
    if (text_len > 0) mx = std::max(mx, st_idx + text_len - 1);
    next_base = mx + 1;
    have_any = true;
    st = ed + lh * lw;
  }
  long long maxpos = have_any ? next_base - 1 : -1;
  if (st < L) {
    const long long st_idx = have_any ? next_base : 0;
    emit_text(st, L - st, st_idx);
    maxpos = st_idx + (L - st) - 1;
  }
  *rope_delta = (int)(maxpos + 1 - L);
  return FO1_OK;
}

}  // namespace fo1

using namespace fo1;

extern "C" int fo1_splice_plan(const int64_t* input_ids, int32_t n_ids, const int32_t* image_grid_hw, int32_t n_images,
                               int32_t n_regions, const fo1_splice_cfg* cfg, int64_t* new_ids, int32_t* src_kind,
                               int32_t* src_index, int32_t* position_ids, int32_t* rope_delta, int32_t* out_len, int32_t capacity) {
  FO1_CHECK_ARG(input_ids && cfg && out_len && rope_delta && n_ids >= 0 && (n_images == 0 || image_grid_hw), "fo1_splice_plan: null argument");
  FO1_CHECK_ARG(cfg->merge > 0, "fo1_splice_plan: merge must be positive");
  std::vector<int64_t> ids;
  std::vector<int> kind, index, pos;
  FO1_TRY(splice_plan(input_ids, n_ids, image_grid_hw, n_images, n_regions, *cfg, ids, kind, index, pos, rope_delta));
  const int L = (int)ids.size();
  *out_len = L;
  if (L > capacity || !new_ids || !src_kind || !src_index || !position_ids) {
    set_error("fo1_splice_plan: capacity %d < required %d", capacity, L);
    return FO1_ERR_WORKSPACE;
  }
  memcpy(new_ids, ids.data(), (size_t)L * sizeof(int64_t));
  memcpy(src_kind, kind.data(), (size_t)L * sizeof(int));
  memcpy(src_index, index.data(), (size_t)L * sizeof(int));
  for (int a = 0; a < 3; ++a) memcpy(position_ids + (size_t)a * capacity, pos.data() + (size_t)a * L, (size_t)L * sizeof(int));
  return FO1_OK;
}

extern "C" int fo1_llm_build_embeds(fo1_model* m, const int32_t* src_kind, const int32_t* src_index, int32_t n_rows,
                                    const void* img_feats, const void* region_feats, void* inputs_embeds, void* stream) {
  FO1_CHECK_ARG(m && src_kind && src_index && inputs_embeds, "fo1_llm_build_embeds: null argument");
  FO1_CHECK_ARG(m->llm.ok, "fo1_llm_build_embeds: model not finalized");
  if (n_rows <= 0) return FO1_OK;
  FO1_CHECK_ARG(m->cfg.llm_hidden % 8 == 0, "fo1_llm_build_embeds: hidden %% 8");
  build_embeds_kernel<<<n_rows, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      src_kind, src_index, m->llm.embed, static_cast<const bf16*>(img_feats), static_cast<const bf16*>(region_feats),
      static_cast<bf16*>(inputs_embeds), m->cfg.llm_hidden);
  FO1_LAUNCH_CHECK();
  return FO1_OK;
}

extern "C" int fo1_llm_generate(fo1_model* m, fo1_generate_desc* d, void* stream) {
  FO1_CHECK_ARG(m && d, "fo1_llm_generate: null argument");
  return llm_generate(m, d, static_cast<cudaStream_t>(stream));
}

extern "C" size_t fo1_decode_attention_workspace_bytes(int32_t n_seqs, int32_t q_heads) {
  return (size_t)(n_seqs > 0 ? n_seqs : 0) * (q_heads > 0 ? q_heads : 0) * fo1::kDecSplits * (128 + 4) * sizeof(float);
}

extern "C" int fo1_decode_attention(const fo1_decode_attn_desc* d, void* stream) {
  using namespace fo1;
  FO1_CHECK_ARG(d != nullptr, "fo1_decode_attention: null descriptor");
  FO1_CHECK_ARG(d->n_seqs >= 0 && d->cap > 0, "fo1_decode_attention: bad n_seqs / cap");
  if (d->n_seqs == 0) return FO1_OK;
  FO1_CHECK_ARG(d->q && d->k_cache && d->v_cache && d->cache_len && d->out, "fo1_decode_attention: null pointer");
  FO1_CHECK_ARG(d->n_seqs <= 65535, "fo1_decode_attention: n_seqs %d exceeds the grid limit", d->n_seqs);
  FO1_CHECK_ARG((d->ldq % 2) == 0 && (d->ldo % 8) == 0 && (reinterpret_cast<uintptr_t>(d->k_cache) & 15) == 0 && (reinterpret_cast<uintptr_t>(d->v_cache) & 15) == 0,
                "fo1_decode_attention: pitches / cache pointers misaligned");
  const size_t need = fo1_decode_attention_workspace_bytes(d->n_seqs, d->q_heads);
  if (d->workspace == nullptr || d->workspace_bytes < need) { set_error("fo1_decode_attention: workspace %zu B < required %zu B", d->workspace_bytes, need); return FO1_ERR_WORKSPACE; }
  return decode_attention(static_cast<const bf16*>(d->q), d->ldq, static_cast<const bf16*>(d->k_cache), static_cast<const bf16*>(d->v_cache), d->cache_len,
                          d->n_seqs, d->cap, d->q_heads, d->kv_heads, d->head_dim, d->scale, static_cast<bf16*>(d->out), d->ldo,
                          static_cast<float*>(d->workspace), static_cast<cudaStream_t>(stream));
}
