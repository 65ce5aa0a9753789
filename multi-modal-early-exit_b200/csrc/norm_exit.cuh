// LayerNorm (+ survivor compaction), attention-bias build, fused exit head / criterion / threshold /
// prefix-sum compaction kernels.
//
//   ln_rows_kernel   : X[dst] = LN(Y[src]) ; dst slot s' <- src slot slot_src[s'] (compaction is free: the
//                      post-LN write goes straight to the survivor's new slot).  HF:300-304, 509-513.
//   bias_build_kernel: (rel_pos + rel_2d_pos)/sqrt(d) + key mask, once per forward, reused by every layer
//                      (EE/models/LayoutLMv3.py:170-179; HF:393-458; mask HF:270-272).
//   exit_fused_kernel: CLS row -> [LN] -> dense/tanh/out_proj (EE/models/LayoutLMv3.py:86-93, 226-227; gate mode
//                      also classifier(CLS) :768) -> logits/T -> max-softmax | entropy (EE_modules.py:149-160)
//                      -> strict threshold test (EE_modules.py:139-143, policy.py:33) -> block prefix-sum over
//                      the fire flags -> survivor list for the next layer, results of leaving documents scattered
//                      to their original document index; one launch per exit, no host round-trip.
#pragma once
#include "embed.cuh"
#include "ptx.cuh"

namespace mmee {

// ------------------------------------------------------------------ ragged row layout of the encoder
// Inside the encoder a document owns only the rows of its KEPT tokens: text tokens with attention_mask != 0 (plus
// token 0, the CLS row every exit reads, even when it is masked as a key) followed by the n_vis visual tokens.  Rows of
// padded text tokens are never computed: nothing reads them (their keys are masked for every query, HF:270-272; exits
// read the CLS row; the mean-pool exits run on the dense embedding output before the encoder).  Slot s of an exit stage
// owns rows [row0[s], row0[s + 1]); row0[n_active] = M is the row count of every GEMM / LayerNorm of the stage.
//   doc_len[doc]      kept text tokens + n_vis                      (keymask_kernel, once per forward)
//   kept_idx[doc][r]  original text position of kept text token r   (keymask_kernel)
//   SlotRows          per exit stage: row0, the attention work list (see attention.cuh) and M
struct SlotRows {
  int* row0;        // [B + 1] exclusive prefix sums of the slots' row counts
  int4* meta;       // [B] {row0, rows, doc, first query tile (prefix of ceil(rows / 128))}  (attention work list)
  int* qt_slot;     // [sum of query tiles] query tile -> slot
  int* n_qt_dev;    // [1] total number of 128-row query tiles
};

// The slot that owns `row`: largest s with row0[s] <= row (row0 ascending, row0[0] = 0, row0[n] = M > row, n >= 1).
// Starts from the proportional guess row * n / M — exact when all documents have the same number of rows (two
// independent loads), a few slots off for ragged batches — and walks from there.
__device__ __forceinline__ int slot_of_row(const int* __restrict__ row0, int n, int M, int row) {
  int s = static_cast<int>(static_cast<float>(row) * (static_cast<float>(n) / static_cast<float>(max(M, 1))));   // a guess: float is fine
  s = max(min(s, n - 1), 0);
  while (__ldg(row0 + s) > row) --s;
  while (__ldg(row0 + s + 1) <= row) ++s;
  return s;
}

// Row plan of one exit stage, by ONE thread block (any blockDim that is a multiple of 32, <= 1024): row0 / meta / qt_slot
// for the n slots whose documents are slot_doc[0 .. n), and the totals.  s_scan: >= 2 * 32 + 2 ints of shared memory.
__device__ __forceinline__ void plan_rows_block(const int* __restrict__ slot_doc, const int* __restrict__ doc_len, int n,
                                                const SlotRows& out, int* __restrict__ m_dev, int q_rows, int* s_scan) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  int* s_w = s_scan;            // [32][2] per-warp totals (rows, query tiles)
  int* s_carry = s_scan + 64;   // [2] running totals
  if (threadIdx.x == 0) { s_carry[0] = 0; s_carry[1] = 0; }
  __syncthreads();
  for (int start = 0; start < n; start += blockDim.x) {
    const int s = start + threadIdx.x;
    const int doc = (s < n) ? slot_doc[s] : 0;
    const int len = (s < n) ? doc_len[doc] : 0;
    const int nq = (len + q_rows - 1) / q_rows;
    int ir = len, iq = nq;                                  // inclusive warp scans
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int tr = __shfl_up_sync(0xffffffffu, ir, o), tq = __shfl_up_sync(0xffffffffu, iq, o);
      if (lane >= o) { ir += tr; iq += tq; }
    }
    if (lane == 31) { s_w[warp * 2] = ir; s_w[warp * 2 + 1] = iq; }
    __syncthreads();
    int br = s_carry[0], bq = s_carry[1];
    for (int w = 0; w < warp; ++w) { br += s_w[w * 2]; bq += s_w[w * 2 + 1]; }
    const int r0 = br + ir - len, q0 = bq + iq - nq;
    if (s < n) {
      out.row0[s] = r0;
      out.meta[s] = make_int4(r0, len, doc, q0);
      for (int k = 0; k < nq; ++k) out.qt_slot[q0 + k] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int tr = 0, tq = 0;
      for (int w = 0; w < nwarps; ++w) { tr += s_w[w * 2]; tq += s_w[w * 2 + 1]; }
      s_carry[0] += tr; s_carry[1] += tq;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out.row0[n] = s_carry[0];
    *out.n_qt_dev = s_carry[1];
    *m_dev = s_carry[0];
  }
}

// stand-alone form (first stage of the encoder, after the embedding-level exits)
__global__ void __launch_bounds__(256) plan_rows_kernel(const int* __restrict__ slot_doc, const int* __restrict__ doc_len,
                                                        const int* __restrict__ n_active_dev, SlotRows out,
                                                        int* __restrict__ m_dev, int q_rows) {
  __shared__ int s_scan[72];
  plan_rows_block(slot_doc, doc_len, *n_active_dev, out, m_dev, q_rows, s_scan);
}

// dense embedding output -> ragged encoder input: dst[row0[s] + r] = src[src_index[s] * seq + token(r)], token(r) = the
// r-th kept text token of the slot's document, then the visual tokens.  `elem_bytes` per element (2: bf16 rows, 4: fp32
// copy of the fp32 engine mode); H * elem_bytes is a multiple of 16.  grid (x, slots).
__global__ void ragged_gather_kernel(const void* __restrict__ src, void* __restrict__ dst,
                                     const int* __restrict__ src_index, const int* __restrict__ slot_doc,
                                     const int* __restrict__ n_active_dev, const int* __restrict__ row0,
                                     const int* __restrict__ doc_len, const int* __restrict__ kept_idx, int n_text,
                                     int n_vis, int seq, int row_bytes) {
  const int slot = blockIdx.y;
  if (slot >= *n_active_dev) return;
  const int doc = slot_doc[slot];
  const int len = doc_len[doc], kept = len - n_vis;
  const int chunks = row_bytes / 16;
  const size_t src_base = static_cast<size_t>(src_index ? src_index[slot] : slot) * seq;
  const size_t dst_base = static_cast<size_t>(row0[slot]);
  const int total = len * chunks;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / chunks, c = i - r * chunks;
    const int tok = (r < kept) ? kept_idx[static_cast<size_t>(doc) * n_text + r] : n_text + (r - kept);
    reinterpret_cast<uint4*>(dst)[(dst_base + r) * chunks + c] = reinterpret_cast<const uint4*>(src)[(src_base + tok) * chunks + c];
  }
}

// one warp per destination row; rows >= *m_dst_dev are skipped.  Xlo (optional): low part of the split-bf16 residual
// stream, Xlo = bf16(v - bf16(v)): the next residual add reads X + Xlo (16-bit mantissa) while the GEMMs read X.
template <int NV>
__global__ void ln_rows_kernel(const float* __restrict__ Y, __nv_bfloat16* __restrict__ X,
                               __nv_bfloat16* __restrict__ Xlo, float* __restrict__ X32, const float* __restrict__ w,
                               const float* __restrict__ b, float eps, int H,
                               const int* __restrict__ m_dst_dev, const int* __restrict__ slot_src,
                               const int* __restrict__ row0_dst, const int* __restrict__ row0_src,
                               const int* __restrict__ n_dst_dev) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= *m_dst_dev) return;
  const int lane = threadIdx.x & 31;
  size_t src_row = row;
  if (slot_src) {                      // survivors of an exit: destination slot s' <- source slot slot_src[s'], same row offset
    const int s = slot_of_row(row0_dst, *n_dst_dev, *m_dst_dev, row);
    src_row = static_cast<size_t>(row0_src[slot_src[s]]) + (row - row0_dst[s]);
  }
  const float* y = Y + src_row * H;
  float v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    v[i] = (c < H) ? y[c] : 0.f;
  }
  warp_layernorm<NV>(v, H, w, b, eps, lane);
  __nv_bfloat16* out = X + static_cast<size_t>(row) * H;
  __nv_bfloat16* out_lo = Xlo ? Xlo + static_cast<size_t>(row) * H : nullptr;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (c < H) {
      const __nv_bfloat16 hi = __float2bfloat16_rn(v[i]);
      out[c] = hi;
      if (out_lo) out_lo[c] = __float2bfloat16_rn(v[i] - __bfloat162float(hi));
      if (X32) X32[static_cast<size_t>(row) * H + c] = v[i];
    }
  }
}

// Vectorised variant for H = 128 * NV4: every lane owns whole float4s (columns 4*(lane + 32*i) .. +3), 16 B loads and
// 8 B stores; two rows per warp iteration keep more loads in flight (the kernel is a pure HBM stream:
// 4 B read + 2 (+2) B written per element).
template <int NV4>
__global__ void __launch_bounds__(256) ln_rows_vec_kernel(const float* __restrict__ Y, __nv_bfloat16* __restrict__ X,
                                                          __nv_bfloat16* __restrict__ Xlo, float* __restrict__ X32,
                                                          const float* __restrict__ w,
                                                          const float* __restrict__ b, float eps, int H,
                                                          const int* __restrict__ m_dst_dev,
                                                          const int* __restrict__ slot_src,
                                                          const int* __restrict__ row0_dst,
                                                          const int* __restrict__ row0_src,
                                                          const int* __restrict__ n_dst_dev,
                                                          float2* __restrict__ stats_out, int* __restrict__ src_out) {
  const int lane = threadIdx.x & 31;
  const int M = *m_dst_dev;
  const int n_dst = slot_src ? *n_dst_dev : 0;
  const int warps_total = gridDim.x * (blockDim.x >> 5);
  float4 w4[NV4], b4[NV4];
#pragma unroll
  for (int i = 0; i < NV4; ++i) {
    w4[i] = __ldg(reinterpret_cast<const float4*>(w + 4 * (lane + 32 * i)));
    b4[i] = __ldg(reinterpret_cast<const float4*>(b + 4 * (lane + 32 * i)));
  }
  // survivors of an exit: destination slot s' <- source slot slot_src[s'], same row offset.  Three dependent loads
  // (row -> slot -> source slot -> its first row): the map of the NEXT row is requested right behind this row's data
  // loads, so the chain resolves under them instead of in front of every row (171 -> 148 us per launch was the gap
  // between the mapped and the unmapped LayerNorm)
  auto map_row = [&](int row) -> size_t {
    if (!slot_src) return static_cast<size_t>(row);
    const int sl = slot_of_row(row0_dst, n_dst, M, row);
    return static_cast<size_t>(__ldg(row0_src + __ldg(slot_src + sl))) + (row - __ldg(row0_dst + sl));
  };
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  size_t next_src = (row < M) ? map_row(row) : 0;
  for (; row < M; row += warps_total) {
    const size_t src_row = next_src;
    const float* y = Y + src_row * H;
    float4 v[NV4];
#pragma unroll
    for (int i = 0; i < NV4; ++i) v[i] = __ldcs(reinterpret_cast<const float4*>(y + 4 * (lane + 32 * i)));   // streamed once
    if (row + warps_total < M) next_src = map_row(row + warps_total);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV4; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    const float mean = warp_sum(s) / H;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
      q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
    }
    const float rstd = rsqrtf(warp_sum(q) / H + eps);
    // "residual from the pre-LayerNorm sums" (gemm.cuh, GemmArgs::resid_y): the next residual add recomputes this row
    // in fp32 from Y[src_row] with these statistics instead of reading a low part
    if (stats_out && lane == 0) {
      stats_out[row] = make_float2(mean, rstd);
      if (src_out) src_out[row] = static_cast<int>(src_row);
    }
    __nv_bfloat16* out = X + static_cast<size_t>(row) * H;
    __nv_bfloat16* out_lo = Xlo ? Xlo + static_cast<size_t>(row) * H : nullptr;
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const float o0 = (v[i].x - mean) * rstd * w4[i].x + b4[i].x, o1 = (v[i].y - mean) * rstd * w4[i].y + b4[i].y;
      const float o2 = (v[i].z - mean) * rstd * w4[i].z + b4[i].z, o3 = (v[i].w - mean) * rstd * w4[i].w + b4[i].w;
      const uint32_t h01 = pack_bf16x2(o0, o1), h23 = pack_bf16x2(o2, o3);
      *reinterpret_cast<uint2*>(out + 4 * (lane + 32 * i)) = make_uint2(h01, h23);
      if (out_lo) {
        const float2 f01 = unpack_bf16x2(h01), f23 = unpack_bf16x2(h23);
        *reinterpret_cast<uint2*>(out_lo + 4 * (lane + 32 * i)) =
            make_uint2(pack_bf16x2(o0 - f01.x, o1 - f01.y), pack_bf16x2(o2 - f23.x, o3 - f23.y));
      }
      if (X32) *reinterpret_cast<float4*>(X32 + static_cast<size_t>(row) * H + 4 * (lane + 32 * i)) = make_float4(o0, o1, o2, o3);
    }
  }
}

// ------------------------------------------------------------------ attention bias
// The additive attention bias (rel_pos + rel_2d_pos)/sqrt(d) is layer-invariant (the reference builds it once per
// forward, EE/models/LayoutLMv3.py:170-179; HF:393-458).  It is materialised once per forward as fp16 in the log2
// domain, bias16[doc][head][i][j] = (W1d[b1] + (Wx[bx] + Wy[by])) * log2(e)/sqrt(d), with -60000 on padded keys
// (attention_mask == 0, HF:270-272) and on the pitch padding j >= seq, so the attention kernel can ADD it on the
// tensor core (S += bias16 x I, see attention.cuh) and needs no separate key mask.  12.3 MB per base document
// instead of 2 x 24 MB fp32 in the reference.
//
// Persistent kernel, one CTA per SM: the 2-D table T2[bx][by][head] = fp16((Wx + Wy) * c) (98 KB for base, built at
// weight load) and T1[b1][head] = W1d * c (fp32) live in shared memory for the whole launch, so each (i, j) pair
// costs one bucket computation for all heads and one T1 + one T2 lookup per head PAIR.
// Row pitch (elements) of the two bias tables in shared memory.  heads % 4 == 0: rows are packed (8 B / 16 B aligned)
// so the kernel reads four heads per LDS.64 / LDS.128; otherwise heads + 2 (an odd number of 32-bit words per fp16 row:
// random rows spread over all banks for the two-head reads).
inline int bias_table_pitch(int heads) { return (heads % 4 == 0) ? heads : heads + 2; }

struct BiasArgs {
  const int64_t* bbox;       // [B, n_text, 4]
  const int* vis_bbox;       // [n_vis, 4]
  const float* t1;           // [bins1][t2_pitch]         W1d * log2(e)/sqrt(d)   (same padded row pitch as t2)
  const __half* t2;          // [bins2*bins2][t2_pitch]   (Wx + Wy) * log2(e)/sqrt(d); row pitch heads + 2 halves = an odd
                             //                           number of 32-bit words, so random rows spread over all smem banks
  const uint8_t* lut1;       // |rel| -> bucket offset, 1-D   (size lut1_n)
  const uint8_t* lut2;       // 2-D
  const float* maskadd;      // [B][kv_pitch] 0 / -inf per key (padding, j >= seq)
  int lut1_n, lut2_n;
  int bins1, bins2;          // rel_pos_bins, rel_2d_pos_bins
  int heads, t2_pitch, n_text, seq, pitch, kv_pitch, B;
  const int* slot_doc;       // survivors of the embedding-level exits: only their documents get a bias (nullptr: all B)
  const int* n_active_dev;
  const int* doc_len;        // [B] kept rows per document (ragged layout: bias rows / columns are indexed by kept-token rank)
  const int* kept_idx;       // [B][n_text] original position of kept text token r
  int n_vis;
  __half* out;               // [B][heads][seq][pitch], indexed by DOCUMENT (the attention kernel maps slot -> doc); only the
                             // first doc_len rows of a document are written, every column j >= doc_len holds the mask value
};

// ragged row r of a document -> original token: kept text token r, or visual token r - kept (index n_text + ...)
__device__ __forceinline__ int bias_token_of_row(const BiasArgs& a, int doc, int len, int r) {
  const int kept = len - a.n_vis;
  return (r < kept) ? a.kept_idx[static_cast<size_t>(doc) * a.n_text + r] : a.n_text + (r - kept);
}

constexpr int BIAS_THREADS = 768;
constexpr float BIAS_MASKED = -60000.0f;   // finite (0 * x stays 0 in the identity MMA) and exp2() of it is 0

inline size_t bias_build_smem(const BiasArgs& a) {
  return static_cast<size_t>(a.bins2) * a.bins2 * a.t2_pitch * 2 + static_cast<size_t>(a.bins1) * a.t2_pitch * 4 + a.lut1_n +
         a.lut2_n + static_cast<size_t>(a.pitch + (a.pitch >> 3) + 8) * 16 + 64;
}

// thread = 8 consecutive keys j of one query row i; a pass covers blockDim / (pitch/8) rows of one document.
__global__ void __launch_bounds__(BIAS_THREADS, 1) bias_build_kernel(BiasArgs a) {
  extern __shared__ __align__(16) uint8_t bsm[];
  const int n_t2 = a.bins2 * a.bins2 * a.t2_pitch;
  __half* s_t2 = reinterpret_cast<__half*>(bsm);
  float* s_t1 = reinterpret_cast<float*>(bsm + static_cast<size_t>(n_t2) * 2);
  // key coordinates, stored at index j + (j >> 3): lane l reads keys 8l .. 8l+7, and the odd stride 9 spreads the
  // warp's 32 reads of "key k of my chunk" over all banks (plain [pitch] arrays gave 8-way conflicts, ncu)
  const int cpitch = a.pitch + (a.pitch >> 3) + 8;
  int* s_pos = reinterpret_cast<int*>(s_t1 + a.bins1 * a.t2_pitch);   // [cpitch] each
  int* s_x = s_pos + cpitch;
  int* s_y = s_x + cpitch;
  int* s_m = s_y + cpitch;                                            // 1 = masked key
  uint8_t* s_l1 = reinterpret_cast<uint8_t*>(s_m + cpitch);
  uint8_t* s_l2 = s_l1 + a.lut1_n;
  for (int i = threadIdx.x; i < n_t2 / 8; i += blockDim.x)
    reinterpret_cast<uint4*>(s_t2)[i] = __ldg(reinterpret_cast<const uint4*>(a.t2) + i);
  for (int i = threadIdx.x; i < a.bins1 * a.t2_pitch; i += blockDim.x) s_t1[i] = a.t1[i];
  for (int i = threadIdx.x; i < a.lut1_n; i += blockDim.x) s_l1[i] = a.lut1[i];
  for (int i = threadIdx.x; i < a.lut2_n; i += blockDim.x) s_l2[i] = a.lut2[i];

  const int chunks = a.pitch >> 3;                      // threads per row
  const int rows_pp = blockDim.x / chunks;              // rows per pass
  const int passes = (a.seq + rows_pp - 1) / rows_pp;   // per document
  const int n_docs = a.n_active_dev ? *a.n_active_dev : a.B;
  const int units = n_docs * passes;
  const int u_lo = static_cast<int>(static_cast<long long>(units) * blockIdx.x / gridDim.x);
  const int u_hi = static_cast<int>(static_cast<long long>(units) * (blockIdx.x + 1) / gridDim.x);
  const int rl = threadIdx.x / chunks;                  // row within the pass
  const int j0 = (threadIdx.x - rl * chunks) * 8;
  const bool active = rl < rows_pp;
  const int half1 = a.bins1 >> 1, half2 = a.bins2 >> 1;
  int cur_doc = -1, cur_len = 0;
  for (int u = u_lo; u < u_hi; ++u) {
    const int dslot = u / passes;
    const int doc = a.slot_doc ? a.slot_doc[dslot] : dslot;
    const int i = (u - dslot * passes) * rows_pp + rl;
    if (doc != cur_doc) {                               // (re)load this document's key coordinates
      __syncthreads();
      cur_len = a.doc_len[doc];
      for (int r = threadIdx.x; r < a.pitch; r += blockDim.x) {
        int pos = 0, x0 = 0, y1 = 0, m = 1;
        if (r < cur_len) {
          const int t = bias_token_of_row(a, doc, cur_len, r);
          if (t < a.n_text) {
            const int64_t* bb = a.bbox + (static_cast<size_t>(doc) * a.n_text + t) * 4;
            pos = t; x0 = static_cast<int>(bb[0]); y1 = static_cast<int>(bb[3]);
          } else {
            const int p = t - a.n_text;
            pos = p; x0 = a.vis_bbox[p * 4 + 0]; y1 = a.vis_bbox[p * 4 + 3];
          }
          m = a.maskadd[static_cast<size_t>(doc) * a.kv_pitch + t] < 0.f ? 1 : 0;    // a kept but masked key: CLS with mask 0
        }
        const int tp = r + (r >> 3);
        s_pos[tp] = pos; s_x[tp] = x0; s_y[tp] = y1; s_m[tp] = m;
      }
      cur_doc = doc;
      __syncthreads();
    }
    if (!active || i >= cur_len) continue;
    const int ip = i + (i >> 3);
    const int pi = s_pos[ip], xi = s_x[ip], yi = s_y[ip];
    const int jp0 = j0 + (j0 >> 3);                    // j0 is a multiple of 8: keys j0 .. j0+7 are contiguous from here
    uint32_t i1[8], i2[8];
    uint32_t mbits = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int j = jp0 + k;
      const int r1 = s_pos[j] - pi, rx = s_x[j] - xi, ry = s_y[j] - yi;
      const int b1 = (r1 > 0 ? half1 : 0) + s_l1[min(abs(r1), a.lut1_n - 1)];
      const int bx = (rx > 0 ? half2 : 0) + s_l2[min(abs(rx), a.lut2_n - 1)];
      const int by = (ry > 0 ? half2 : 0) + s_l2[min(abs(ry), a.lut2_n - 1)];
      i1[k] = static_cast<uint32_t>(b1 * a.t2_pitch);
      i2[k] = static_cast<uint32_t>((bx * a.bins2 + by) * a.t2_pitch);
      mbits |= static_cast<uint32_t>(s_m[j]) << k;
    }
    __half* out = a.out + ((static_cast<size_t>(doc) * a.heads) * a.seq + i) * a.pitch + j0;
    const size_t head_stride = static_cast<size_t>(a.seq) * a.pitch;
    // the 1-D buckets are log-spaced: away from the diagonal all 8 keys of a chunk share one, and that table row is
    // read once per head pair instead of once per key
    bool same1 = true;
#pragma unroll
    for (int k = 1; k < 8; ++k) same1 = same1 && (i1[k] == i1[0]);
    auto pack = [](float lo, float hi) {
      __half2 t = __floats2half2_rn(lo, hi);
      return *reinterpret_cast<uint32_t*>(&t);
    };
    if ((a.heads & 3) == 0) {
      // table rows are 8 B (fp16) / 16 B (fp32) aligned: four heads per shared-memory read
      for (int h = 0; h < a.heads; h += 4) {
        float v[4][8];
        const float4 t1c = *reinterpret_cast<const float4*>(s_t1 + i1[0] + h);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float4 t1 = t1c;
          if (!same1) t1 = *reinterpret_cast<const float4*>(s_t1 + i1[k] + h);
          const uint2 raw = *reinterpret_cast<const uint2*>(s_t2 + i2[k] + h);
          const float2 ta = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
          const float2 tb = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
          v[0][k] = t1.x + ta.x; v[1][k] = t1.y + ta.y; v[2][k] = t1.z + tb.x; v[3][k] = t1.w + tb.y;
        }
        if (mbits) {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            if ((mbits >> k) & 1u) { v[0][k] = BIAS_MASKED; v[1][k] = BIAS_MASKED; v[2][k] = BIAS_MASKED; v[3][k] = BIAS_MASKED; }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          *reinterpret_cast<uint4*>(out + (h + q) * head_stride) =
              make_uint4(pack(v[q][0], v[q][1]), pack(v[q][2], v[q][3]), pack(v[q][4], v[q][5]), pack(v[q][6], v[q][7]));
      }
      continue;
    }
    for (int h = 0; h < a.heads; h += 2) {
      float v0[8], v1[8];
      float2 t1c = *reinterpret_cast<const float2*>(s_t1 + i1[0] + h);
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float2 t1 = t1c;
        if (!same1) t1 = *reinterpret_cast<const float2*>(s_t1 + i1[k] + h);
        const float2 t2 = __half22float2(*reinterpret_cast<const __half2*>(s_t2 + i2[k] + h));
        v0[k] = t1.x + t2.x;
        v1[k] = t1.y + t2.y;
      }
      if (mbits) {                                     // padded keys (rare): the mask rides in the bias
#pragma unroll
        for (int k = 0; k < 8; ++k)
          if ((mbits >> k) & 1u) { v0[k] = BIAS_MASKED; v1[k] = BIAS_MASKED; }
      }
      *reinterpret_cast<uint4*>(out + h * head_stride) =
          make_uint4(pack(v0[0], v0[1]), pack(v0[2], v0[3]), pack(v0[4], v0[5]), pack(v0[6], v0[7]));
      *reinterpret_cast<uint4*>(out + (h + 1) * head_stride) =
          make_uint4(pack(v1[0], v1[1]), pack(v1[2], v1[3]), pack(v1[4], v1[5]), pack(v1[6], v1[7]));
    }
  }
}

// fp32 engine mode: the same bias as a split-fp16 pair (hi + lo carries 22 mantissa bits), from fp32 tables
// T1[b1][head], TX[bx][head], TY[by][head] (each already times log2(e)/sqrt(d); 8 KB together, L1-resident) instead of
// the fp16 2-D table: v = T1 + (TX + TY) in fp32 as the reference sums them (HF:416-458), hi = fp16(v), lo = fp16(v - hi).
// Not on the throughput path: one thread per (query row, 8 keys), grid.y = survivor slot.
__global__ void bias_build_split_kernel(BiasArgs a, const float* __restrict__ tx, const float* __restrict__ ty,
                                        __half* __restrict__ out_lo) {
  const int dslot = blockIdx.y;
  if (dslot >= (a.n_active_dev ? *a.n_active_dev : a.B)) return;
  const int doc = a.slot_doc ? a.slot_doc[dslot] : dslot;
  const int chunks = a.pitch >> 3;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int len = a.doc_len[doc];
  if (idx >= len * chunks) return;
  const int i = idx / chunks, j0 = (idx - i * chunks) * 8;
  auto coords = [&](int r, int& pos, int& x0, int& y1, int& t) {
    t = bias_token_of_row(a, doc, len, r);
    if (t < a.n_text) {
      const int64_t* bb = a.bbox + (static_cast<size_t>(doc) * a.n_text + t) * 4;
      pos = t; x0 = static_cast<int>(bb[0]); y1 = static_cast<int>(bb[3]);
    } else {
      const int p = t - a.n_text;
      pos = p; x0 = a.vis_bbox[p * 4 + 0]; y1 = a.vis_bbox[p * 4 + 3];
    }
  };
  int pi, xi, yi, ti;
  coords(i, pi, xi, yi, ti);
  const int half1 = a.bins1 >> 1, half2 = a.bins2 >> 1;
  int i1[8], ix[8], iy[8];
  bool masked[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int j = j0 + k;
    masked[k] = true;
    i1[k] = ix[k] = iy[k] = 0;
    if (j < len) {
      int pj, xj, yj, tj;
      coords(j, pj, xj, yj, tj);
      const int r1 = pj - pi, rx = xj - xi, ry = yj - yi;
      i1[k] = ((r1 > 0 ? half1 : 0) + a.lut1[min(abs(r1), a.lut1_n - 1)]) * a.t2_pitch;
      ix[k] = ((rx > 0 ? half2 : 0) + a.lut2[min(abs(rx), a.lut2_n - 1)]) * a.t2_pitch;
      iy[k] = ((ry > 0 ? half2 : 0) + a.lut2[min(abs(ry), a.lut2_n - 1)]) * a.t2_pitch;
      masked[k] = a.maskadd[static_cast<size_t>(doc) * a.kv_pitch + tj] < 0.f;
    }
  }
  const size_t head_stride = static_cast<size_t>(a.seq) * a.pitch;
  const size_t base = ((static_cast<size_t>(doc) * a.heads) * a.seq + i) * a.pitch + j0;
  for (int h = 0; h < a.heads; ++h) {
    __align__(16) __half hi[8], lo[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float v = __ldg(a.t1 + i1[k] + h) + (__ldg(tx + ix[k] + h) + __ldg(ty + iy[k] + h));
      if (masked[k]) v = BIAS_MASKED;
      hi[k] = __float2half_rn(v);
      lo[k] = masked[k] ? __float2half_rn(0.f) : __float2half_rn(v - __half2float(hi[k]));
    }
    *reinterpret_cast<uint4*>(a.out + base + h * head_stride) = *reinterpret_cast<const uint4*>(hi);
    *reinterpret_cast<uint4*>(out_lo + base + h * head_stride) = *reinterpret_cast<const uint4*>(lo);
  }
}

// Key-padding mask (HF:270-272 adds (1-mask)*finfo.min to the scores): maskadd[doc][t] = 0 / -inf per ORIGINAL token
// position, and the document's kept-token list for the ragged encoder layout: kept_idx[doc][r] = position of the r-th
// text token with attention_mask != 0 (token 0, the CLS row every exit reads, is always kept), doc_len[doc] = kept text
// tokens + n_vis.  grid B, block = kv_pitch threads (<= 1024, a multiple of 32).
__global__ void keymask_kernel(const int64_t* __restrict__ mask, float* __restrict__ maskadd, int* __restrict__ kept_idx,
                               int* __restrict__ doc_len, int n_text, int seq, int kv_pitch) {
  __shared__ int s_w[33];
  const int doc = blockIdx.x;
  const int j = threadIdx.x;
  const int lane = j & 31, warp = j >> 5, nwarps = blockDim.x >> 5;
  bool m = (j >= seq);
  if (!m && j < n_text) m = (mask[static_cast<size_t>(doc) * n_text + j] == 0);
  if (j < kv_pitch) maskadd[static_cast<size_t>(doc) * kv_pitch + j] = m ? -INFINITY : 0.f;
  const int keep = (j < n_text) && (!m || j == 0);
  int incl = keep;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const int v = (lane < nwarps) ? s_w[lane] : 0;
    int wi = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    s_w[lane] = wi - v;                          // exclusive warp offsets
    if (lane == 31) s_w[32] = wi;                // kept text tokens of the document
  }
  __syncthreads();
  if (keep) kept_idx[static_cast<size_t>(doc) * n_text + s_w[warp] + incl - 1] = j;
  if (j == 0) doc_len[doc] = s_w[32] + (seq - n_text);
}

// ------------------------------------------------------------------ exit head
struct HeadWeights {
  const float* dense_w;   // [H, H] or nullptr (1-layer head)
  const float* dense_b;   // [H]
  const float* out_w;     // [n_out, H]
  const float* out_b;     // [n_out]
  int n_out;
};

// out_proj of one row: y[j] = w[j] . x + b[j] for j < n_out (<= 32); lane j returns y[j].  Eight outputs at a time so
// that eight independent weight loads are in flight per step (one dot after the other left a single L2 round trip
// outstanding per step, and the 18 dots of a gate-mode exit took most of the kernel's 50 us).
__device__ __forceinline__ float warp_dots_to_lanes(const float* __restrict__ w, const float* __restrict__ b,
                                                    const float* __restrict__ x, int H, int n_out, int lane) {
  float mine = 0.f;
  for (int j0 = 0; j0 < n_out; j0 += 8) {
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int k = lane * 4; k < H; k += 128) {
      const float4 x4 = *reinterpret_cast<const float4*>(x + k);
      float4 w4[8];
#pragma unroll
      for (int j = 0; j < 8; ++j)
        w4[j] = (j0 + j < n_out) ? __ldg(reinterpret_cast<const float4*>(w + static_cast<size_t>(j0 + j) * H + k))
                                 : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        acc[j] = fmaf(w4[j].x, x4.x, acc[j]);
        acc[j] = fmaf(w4[j].y, x4.y, acc[j]);
        acc[j] = fmaf(w4[j].z, x4.z, acc[j]);
        acc[j] = fmaf(w4[j].w, x4.w, acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float v = warp_sum(acc[j]);
      if (lane == j0 + j) mine = v + __ldg(b + j0 + j);
    }
  }
  return mine;
}

// ------------------------------------------------------------------ compaction
struct CompactArgs {
  const int* n_active_dev;     // current number of active slots
  int* n_next_dev;             // out: survivors
  int* m_next_dev;             // out: survivors * seq  (row count for the next layer's GEMMs)
  int seq;
  const int* slot_doc;         // [n] slot -> original document index
  int* next_slot_doc;          // [n_next]
  int* next_slot_src;          // [n_next] new slot -> old slot (row gather map for the LN that follows)
  const int* slot_fire;
  const float* slot_logits;    // [n, K]
  const float* slot_head;      // [n, n_head]
  const float* slot_crit;
  int K, n_head;
  int exit_index;              // e
  int leave;                   // 1: firing documents leave (early-exit mode); 0: dense mode, everyone stays
  // per-document outputs
  float* out_logits;           // [B, K]
  float* out_crit;             // [B]
  int* out_exit;               // [B]  (-1 = undecided)
  float* all_logits;           // [(E+1), B, K] or nullptr
  float* all_head;             // [(E+1), B, n_head_max] or nullptr
  float* all_crit;             // [(E+1), B] or nullptr
  int B, n_head_max;
  unsigned long long* hist;    // [E+1]
  // row plan of the next stage (ragged layout)
  const int* doc_len;          // [B]
  SlotRows next_rows;
  int q_rows;                  // query rows per attention item (128)
};

// ------------------------------------------------------------------ fused exit stage (one launch per exit)
// exit_fused_kernel: CLS rows + LayerNorm, dense + tanh, out_proj + criterion + threshold, and the survivor compaction
// in ONE launch.  CTA (fb, g, job): documents 16g..16g+15 of the active slots, dense features
// 32fb..32fb+31 of head `job`:
//   1. LayerNorm of the group's CLS rows into shared memory (fp32, two-pass; redundant per feature block: cheap);
//   2. warp = 4 features x 16 documents: W rows streamed from L2 (float4), Z from smem, fp32 FMA, butterfly
//      reduction over the K-split lanes, T = tanh(. + b) to global scratch;
//   3. the LAST CTA of a group to finish (atomic ticket) runs out_proj / temperature / criterion / strict threshold
//      for its 16 documents 
//   4. the LAST group to finish runs the prefix-sum compaction over all active slots (compact logic).
// No host round-trip and no extra launches: ~4x fewer launches and no exposed load latency between the stages.
struct ExitFusedArgs {
  // (1) rows
  const float* rows;        // fp32 rows; row of slot s starts at rows + src(s) * row_stride, or, with row_off (ragged
  size_t row_stride;        // encoder layout: the slot's CLS row is its first row), at rows + row_off[src(s)] * H
  const int* row_off;
  const int* slot_src;      // optional gather map (rows not yet compacted)
  const float* ln_w;        // nullptr -> no LayerNorm (mean-pooled embedding exit)
  const float* ln_b;
  float ln_eps;
  int H;
  const int* n_active_dev;
  // (2) dense jobs
  int jobs;                 // 0..2
  const float* w[2];        // [H, H]
  const float* b[2];
  float* T[2];              // [maxB, H] scratch
  // (3) heads: input of each out_proj: 0 / 1 = T[0] / T[1], 2 = the normalised rows themselves, -1 = head unused
  int head_src, cls_src;
  HeadWeights head, cls;
  int gate_mode, n_labels, criterion;   // criterion: 0 max softmax (>), 1 entropy (<), 2 LTE (<)
  const float* lte_w;       // criterion 2: the learned-to-exit scorer sigmoid(lte_w . row + lte_b) on the exit head's
  float lte_b;              // own input row (EE/models/LayoutLMv3.py:142-149, 231-237); the class logits are unchanged
  float* slot_lte;          // [maxB] scratch
  float inv_temp, threshold;
  const float* policy;      // optional (captured forward plans): {threshold, 1/T} of this exit in device memory, read
                            // instead of the two scalars above so that one graph serves every policy
  int force;
  // optional (captured forward plans, early-exit mode): the compacting thread sets this IF-node condition to
  // "someone survived", so the launches of the deeper layers are skipped once every document has left
  cudaGraphConditionalHandle cond;
  int set_cond;
  float* slot_logits; float* slot_head; float* slot_crit; int* slot_fire;
  // tickets (zero on entry, reset by the last arriver)
  unsigned int* group_ticket;   // [ceil(maxB/16)]
  unsigned int* groups_done;    // [1]
  // (4)
  CompactArgs compact;
};

constexpr int EXF_DOCS = 16, EXF_FEATS = 32, EXF_THREADS = 256;

inline size_t exit_fused_smem(int H) { return static_cast<size_t>(2) * EXF_DOCS * H * sizeof(float) + 64; }

// block-wide compaction (any blockDim that is a multiple of 32, <= 1024); loads of this launch's results bypass L1
__device__ __forceinline__ void compact_block(const CompactArgs& a, int* s_warp, int* s_misc) {
  int& s_total = s_misc[0];
  int& s_base = s_misc[1];
  int& s_fired = s_misc[2];
  const int n = *a.n_active_dev;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  if (threadIdx.x == 0) { s_base = 0; s_fired = 0; }
  __syncthreads();
  for (int start = 0; start < n; start += blockDim.x) {
    const int s = start + threadIdx.x;
    const bool valid = s < n;
    int doc = -1, fire = 0, first = 0;
    if (valid) {
      doc = a.slot_doc[s];
      fire = __ldcg(a.slot_fire + s);
      if (a.all_logits)
        for (int k = 0; k < a.K; ++k)
          a.all_logits[(static_cast<size_t>(a.exit_index) * a.B + doc) * a.K + k] = __ldcg(a.slot_logits + static_cast<size_t>(s) * a.K + k);
      if (a.all_head)
        for (int k = 0; k < a.n_head; ++k)
          a.all_head[(static_cast<size_t>(a.exit_index) * a.B + doc) * a.n_head_max + k] = __ldcg(a.slot_head + static_cast<size_t>(s) * a.n_head + k);
      if (a.all_crit) a.all_crit[static_cast<size_t>(a.exit_index) * a.B + doc] = __ldcg(a.slot_crit + s);
      first = fire && (a.out_exit[doc] < 0);
      if (first) {
        a.out_exit[doc] = a.exit_index;
        a.out_crit[doc] = __ldcg(a.slot_crit + s);
        for (int k = 0; k < a.K; ++k) a.out_logits[static_cast<size_t>(doc) * a.K + k] = __ldcg(a.slot_logits + static_cast<size_t>(s) * a.K + k);
      }
    }
    const int stay = valid && !(a.leave && fire);
    const unsigned ball = __ballot_sync(0xffffffffu, stay);
    const int wprefix = __popc(ball & ((1u << lane) - 1));
    const unsigned fball = __ballot_sync(0xffffffffu, first);
    if (lane == 0) { s_warp[warp] = __popc(ball); if (fball) atomicAdd(&s_fired, __popc(fball)); }
    __syncthreads();
    if (warp == 0) {
      const int v = (lane < nwarps) ? s_warp[lane] : 0;
      int incl = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
      s_warp[lane] = incl - v;                 // exclusive per-warp offsets
      if (lane == 31) s_total = incl;
    }
    __syncthreads();
    if (stay) {
      const int dst = s_base + s_warp[warp] + wprefix;
      a.next_slot_doc[dst] = doc;
      a.next_slot_src[dst] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base += s_total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    *a.n_next_dev = s_base;
    if (s_fired) atomicAdd(a.hist + a.exit_index, static_cast<unsigned long long>(s_fired));
  }
  __syncthreads();
  // rows of the survivors: row0 / attention work list / M of the next stage (next_slot_doc was written by this block)
  __shared__ int s_scan[72];
  const int n_next = s_base;
  __threadfence_block();
  plan_rows_block(a.next_slot_doc, a.doc_len, n_next, a.next_rows, a.m_next_dev, a.q_rows, s_scan);
}

__global__ void __launch_bounds__(EXF_THREADS) exit_fused_kernel(ExitFusedArgs a) {
  extern __shared__ __align__(16) float exf_smem[];
  __shared__ int s_warp[32];
  __shared__ int s_misc[4];
  __shared__ unsigned int s_ticket;
  const int H = a.H;
  float* sZ = exf_smem;                         // [16][H] normalised rows; later the head's out_proj input
  float* sX = exf_smem + EXF_DOCS * H;          // [16][H] the classifier's out_proj input (gate mode)
  const int n = *a.n_active_dev;
  const int n_groups = (n + EXF_DOCS - 1) / EXF_DOCS;
  const int g = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (n == 0) {                                 // nobody left: still publish the (empty) survivor list
    if (blockIdx.x == 0 && g == 0 && blockIdx.z == 0) {
      compact_block(a.compact, s_warp, s_misc);
      if (a.set_cond && threadIdx.x == 0) cudaGraphSetConditional(a.cond, 0u);
    }
    return;
  }
  if (g >= n_groups) return;
  const int d0 = g * EXF_DOCS;

  // ---- (1) rows of this group -> sZ (LayerNorm unless this is the pooled embedding exit)
  for (int dd = warp; dd < EXF_DOCS; dd += EXF_THREADS / 32) {
    const int slot = d0 + dd;
    float* z = sZ + dd * H;
    if (slot >= n) {
      for (int c = lane * 4; c < H; c += 128) *reinterpret_cast<float4*>(z + c) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    const int src = a.slot_src ? a.slot_src[slot] : slot;
    const float* r = a.row_off ? a.rows + static_cast<size_t>(a.row_off[src]) * H : a.rows + static_cast<size_t>(src) * a.row_stride;
    float4 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = (lane + 32 * i) * 4;
      v[i] = (c < H) ? *reinterpret_cast<const float4*>(r + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (a.ln_w) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      const float mean = warp_sum(s) / H;
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if ((lane + 32 * i) * 4 < H) {
          const float dx = v[i].x - mean, dy = v[i].y - mean, dz = v[i].z - mean, dw = v[i].w - mean;
          q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
        }
      }
      const float rstd = rsqrtf(warp_sum(q) / H + a.ln_eps);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (c < H) {
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(a.ln_w + c));
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(a.ln_b + c));
          v[i].x = (v[i].x - mean) * rstd * w4.x + b4.x;
          v[i].y = (v[i].y - mean) * rstd * w4.y + b4.y;
          v[i].z = (v[i].z - mean) * rstd * w4.z + b4.z;
          v[i].w = (v[i].w - mean) * rstd * w4.w + b4.w;
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = (lane + 32 * i) * 4;
      if (c < H) *reinterpret_cast<float4*>(z + c) = v[i];
    }
    if (a.lte_w && blockIdx.x == 0 && blockIdx.z == 0) {       // one CTA of the group scores the rows
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = (lane + 32 * i) * 4;
        if (c < H) {
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(a.lte_w + c));
          acc = fmaf(w4.x, v[i].x, acc); acc = fmaf(w4.y, v[i].y, acc);
          acc = fmaf(w4.z, v[i].z, acc); acc = fmaf(w4.w, v[i].w, acc);
        }
      }
      acc = warp_sum(acc);
      if (lane == 0) a.slot_lte[slot] = acc + a.lte_b;
    }
  }
  __syncthreads();

  // ---- (2) dense + tanh: warp = 4 features x 16 documents, lanes split K
  if (a.jobs > 0) {
    const int job = blockIdx.z;
    const int f0 = blockIdx.x * EXF_FEATS + warp * 4;
    const float* __restrict__ W = a.w[job] + static_cast<size_t>(f0) * H;
    float acc[64];
#pragma unroll
    for (int i = 0; i < 64; ++i) acc[i] = 0.f;
    float4 wn[4];                                 // weights of the NEXT k step: its L2 round trip overlaps this step's FMAs
#pragma unroll
    for (int f = 0; f < 4; ++f) wn[f] = __ldg(reinterpret_cast<const float4*>(W + static_cast<size_t>(f) * H + lane * 4));
    for (int k = lane * 4; k < H; k += 128) {
      float4 w4[4];
#pragma unroll
      for (int f = 0; f < 4; ++f) w4[f] = wn[f];
      if (k + 128 < H) {
#pragma unroll
        for (int f = 0; f < 4; ++f) wn[f] = __ldg(reinterpret_cast<const float4*>(W + static_cast<size_t>(f) * H + k + 128));
      }
#pragma unroll
      for (int d = 0; d < EXF_DOCS; ++d) {
        const float4 z4 = *reinterpret_cast<const float4*>(sZ + d * H + k);
#pragma unroll
        for (int f = 0; f < 4; ++f) {
          float t = acc[f * 16 + d];
          t = fmaf(w4[f].x, z4.x, t); t = fmaf(w4[f].y, z4.y, t); t = fmaf(w4[f].z, z4.z, t); t = fmaf(w4[f].w, z4.w, t);
          acc[f * 16 + d] = t;
        }
      }
    }
    // butterfly reduction over the 32 K-split lanes: halves the live values per step; lane ends with indices 2*lane, 2*lane+1
#pragma unroll
    for (int off = 16, cnt = 64; off >= 1; off >>= 1, cnt >>= 1) {
      const bool up = (lane & off) != 0;
#pragma unroll
      for (int j = 0; j < cnt / 2; ++j) {
        const float send = up ? acc[j] : acc[j + cnt / 2];
        const float keep = up ? acc[j + cnt / 2] : acc[j];
        acc[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = 2 * lane + j, f = idx >> 4, d = idx & 15;
      if (d0 + d < n)
        a.T[job][static_cast<size_t>(d0 + d) * H + f0 + f] = tanhf(acc[j] + __ldg(a.b[job] + f0 + f));
    }
  }

  // ---- ticket: the last CTA of this group continues with the heads
  __threadfence();
  __syncthreads();
  const unsigned int per_group = gridDim.x * gridDim.z;
  if (threadIdx.x == 0) s_ticket = atomicAdd(a.group_ticket + g, 1u);
  __syncthreads();
  if (s_ticket != per_group - 1) return;
  if (threadIdx.x == 0) a.group_ticket[g] = 0u;            // ready for the next exit
  __threadfence();

  // ---- (3) out_proj inputs into shared memory (T rows were written by other SMs: bypass L1)
  const int K = a.n_labels;
  const float inv_temp = a.policy ? a.policy[1] : a.inv_temp;
  const float threshold = a.policy ? a.policy[0] : a.threshold;
  if (a.head_src == 0 || a.head_src == 1) {
    const float* Tsrc = a.T[a.head_src];
    for (int i = threadIdx.x; i < EXF_DOCS * H / 4; i += EXF_THREADS) {
      const int d = (i * 4) / H;
      reinterpret_cast<float4*>(sZ)[i] = (d0 + d < n) ? __ldcg(reinterpret_cast<const float4*>(Tsrc + static_cast<size_t>(d0) * H) + i)
                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  if (a.gate_mode) {
    const float* Tsrc = a.T[a.cls_src];
    for (int i = threadIdx.x; i < EXF_DOCS * H / 4; i += EXF_THREADS) {
      const int d = (i * 4) / H;
      reinterpret_cast<float4*>(sX)[i] = (d0 + d < n) ? __ldcg(reinterpret_cast<const float4*>(Tsrc + static_cast<size_t>(d0) * H) + i)
                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  __syncthreads();
  for (int dd = warp; dd < EXF_DOCS; dd += EXF_THREADS / 32) {
    const int slot = d0 + dd;
    if (slot >= n) continue;
    float head_val = 0.f;                 // lane j holds head logit j
    if (a.head_src >= 0 && a.head.out_w) {
      head_val = warp_dots_to_lanes(a.head.out_w, a.head.out_b, sZ + dd * H, H, a.head.n_out, lane);
      if (lane < a.head.n_out) a.slot_head[static_cast<size_t>(slot) * a.head.n_out + lane] = head_val;
    }
    float raw = head_val;                 // class logit of lane k
    if (a.gate_mode) raw = warp_dots_to_lanes(a.cls.out_w, a.cls.out_b, sX + dd * H, H, K, lane);
    if (lane < K) a.slot_logits[static_cast<size_t>(slot) * K + lane] = raw;
    const float z = raw * inv_temp;
    const float zmax = warp_max(lane < K ? z : -INFINITY);
    const float ex = (lane < K) ? expf(z - zmax) : 0.f;
    const float A = warp_sum(ex);
    float crit;
    if (a.criterion == 0) {
      crit = 1.0f / A;
    } else if (a.criterion == 2) {
      crit = 1.0f / (1.0f + expf(-__ldcg(a.slot_lte + slot)));     // nn.Sigmoid of the LTE score (written by another SM)
    } else {
      const float Bz = warp_sum((lane < K) ? (z - zmax) * ex : 0.f);
      crit = logf(A) - Bz / A;
    }
    if (lane == 0) {
      a.slot_crit[slot] = crit;
      const bool fire = a.force || (a.criterion == 0 ? (crit > threshold) : (crit < threshold));
      a.slot_fire[slot] = fire ? 1 : 0;
    }
  }

  // ---- (4) the last group to finish compacts
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_ticket = atomicAdd(a.groups_done, 1u);
  __syncthreads();
  if (s_ticket != static_cast<unsigned int>(n_groups) - 1) return;
  if (threadIdx.x == 0) *a.groups_done = 0u;
  __threadfence();
  compact_block(a.compact, s_warp, s_misc);
  if (a.set_cond && threadIdx.x == 0) cudaGraphSetConditional(a.cond, s_misc[1] > 0 ? 1u : 0u);   // s_misc[1]: survivors
}

}  // namespace mmee
