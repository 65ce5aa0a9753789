// Persistent warp-specialised tcgen05 GEMM for sm_100a:  C[M,N] = A[M,K] * W[N,K]^T (+ fused epilogue).
//
//   A  : activations, bf16 row-major [M_max, K]   (TMA, 128 x 64 boxes, SWIZZLE_128B)
//   W  : nn.Linear weight, bf16 row-major [N, K]  (TMA, BLOCK_N x 64 boxes, SWIZZLE_128B)
//   acc: fp32 in TMEM, 2 accumulator buffers of BLOCK_N columns (epilogue of tile i overlaps MMA of i+1)
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer (one elected lane),
// warps 2..9 = epilogue (TMEM lane quarter = warp % 4, column half = (warp-2)/4); each warp transposes its
// 32x32 chunk through a private swizzled smem slab so global stores are row-contiguous (coalesced).  M (the surviving-token count) is read from
// device memory so the grid never depends on a host round-trip: grid = #SMs, static round-robin tiles.
//
// SPLIT (fp32 engine mode): every operand is a split-bf16 pair (hi = bf16(v), lo = bf16(v - hi): 16 mantissa bits) and
// the k loop runs three segments into the same fp32 accumulator: A_hi W_hi^T + A_lo W_hi^T + A_hi W_lo^T (the lo x lo
// term is below 2^-18 relative and dropped).  Same tiles, same pipeline, three times the MMAs; bf16 outputs are written
// as (hi, lo) pairs too.  Logit error vs the fp32 reference drops from ~3e-3 to ~5e-6 (tests, DESIGN.md).
//
// Replaces the nn.Linear call sites of HF LayoutLMv3 used by the reference: query/key/value
// (HF modeling_layoutlmv3.py:245-259), SelfOutput.dense (:300-304), Intermediate.dense + GELU
// (:495-498), Output.dense (:509-513), and the patch-embedding conv as a GEMM (:70-82).
#pragma once
#include <cuda.h>

#include "ptx.cuh"
#include "tmap.h"

namespace mmee {

constexpr int GEMM_BLOCK_M = 128;
constexpr int GEMM_BLOCK_K = 64;
constexpr int GEMM_EPI_WARPS = 8;                    // two warps per TMEM lane quarter (column halves)
constexpr int GEMM_THREADS = 64 + GEMM_EPI_WARPS * 32;

enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,   // out_bf16[m, n] = acc + bias[n]
  EPI_GELU_BF16 = 1,   // out_bf16[m, n] = gelu_erf(acc + bias[n])
  EPI_RESID_F32 = 2,   // out_f32 [m, n] = acc + bias[n] + resid_bf16[m, n] (+ resid_lo_bf16[m, n])  |  + LayerNorm(resid_y[src(m)])[n]
  EPI_QKV = 3,         // n < qk_cols: qk_bf16[m, n];  else V^T: vt[doc][head][d][kv_pitch]
  EPI_PATCH = 4,       // patch-embed rows (doc*n_patch + p): out_f32[(doc*n_vis + 1 + p), n] = acc + bias + pos[1+p, n]
};

struct GemmArgs {
  const int* m_dev;        // device pointer to the dynamic row count (nullptr -> m_static)
  int m_static;
  int N, K;
  const float* bias;       // [N]
  void* out;               // bf16 or f32 [*, ld_out]
  __nv_bfloat16* out_lo;   // SPLIT: low parts of a bf16 output (same layout as out)
  int ld_out;
  const __nv_bfloat16* resid;   // EPI_RESID_F32: [*, N]
  const __nv_bfloat16* resid_lo;   // optional low part of a split-bf16 residual (resid + resid_lo = 16-bit mantissa), or nullptr
  const float* resid_f32;          // fp32 engine mode: the residual itself in fp32 (exact, as the reference adds it); replaces resid / resid_lo
  // bf16 mode, "residual from the pre-LayerNorm sums": the residual of output row r is LayerNorm(resid_y[src(r)]),
  // recomputed here in fp32 from the sums the LayerNorm kernel read (it left mean / rstd per row), so that kernel
  // writes no low part and the residual is exact.  Replaces resid / resid_lo when resid_y != nullptr.
  const float* resid_y;            // [*, N] fp32 pre-LayerNorm sums (never the buffer `out` points to)
  const float2* resid_stats;       // [rows] (mean, rstd) of output row r's residual row
  const int* resid_src;            // [rows] row of resid_y behind output row r (an exit compaction in between), nullptr: r
  const float* resid_w;            // [N] LayerNorm weight / bias of that LayerNorm
  const float* resid_b;
  int resid_prefetch;              // pair kernel: pull the next tile's rows of resid_y into L2 while this tile's MMAs run
  // EPI_QKV
  __nv_bfloat16* vt;       // [docs][heads][64][kv_pitch]
  __nv_bfloat16* vt_lo;    // SPLIT: low parts of V^T
  int qk_cols;             // 2*H
  const int* row0;         // [n_slots + 1] first row of every slot (ragged documents); V^T is indexed by (slot, row - row0)
  const int* n_slots_dev;
  int kv_pitch;            // padded token pitch of V^T rows
  int heads;
  // EPI_PATCH
  const float* pos;        // pos_embed [n_vis, N]
  int n_patch, n_vis;
};

template <int BLOCK_N>
struct GemmSmem {
  static constexpr int STAGES = (BLOCK_N == 256) ? 4 : 6;
  static constexpr int A_BYTES = GEMM_BLOCK_M * GEMM_BLOCK_K * 2;
  static constexpr int B_BYTES = BLOCK_N * GEMM_BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STG_OFF = STAGES * STAGE_BYTES;             // per-warp 32 x 128 B transpose staging
  static constexpr int BAR_OFF = STG_OFF + GEMM_EPI_WARPS * 4096;
  static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 4) * 8 + 16;
  static constexpr int DYN_BYTES = TOTAL + 1024;   // slack for manual 1024 B alignment
};

__device__ __forceinline__ float gelu_erf_fast(float x) {
  // x * Phi(x) with Phi(x) = 1 - 0.5*erfc(x/sqrt2) for x >= 0 and 0.5*erfc(|x|/sqrt2) for x < 0.
  // 0.5*erfc(z) = 2^q(z), q a degree-6 minimax fit of log2(0.5*erfc(z)) on z in [0, 4.3] (|abs err| < 4.2e-7 on
  // 0.5*erfc, fitted offline; beyond z = 4.3 erfc < 2e-9 and the clamp keeps it there): matches torch's exact-erf
  // GELU (activations.py "gelu" -> nn.functional.gelu) to 2.3e-7 absolute, far inside the bf16 rounding of the
  // output.  1 MUFU (ex2) + 11 FMA/ALU-pipe ops (the A&S 7.1.26 form needed 2 MUFU + ~15).
  const float z = fminf(fabsf(x) * 0.70710678118654752f, 4.3f);
  float q = 2.699725252e-04f;
  q = fmaf(q, z, -4.347565948e-03f);
  q = fmaf(q, z, 3.221176717e-02f);
  q = fmaf(q, z, -1.508187237e-01f);
  q = fmaf(q, z, -9.177533792e-01f);
  q = fmaf(q, z, -1.627978526e+00f);
  q = fmaf(q, z, -9.999988147e-01f);
  float h;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(h) : "f"(q));        // 0.5 * erfc(|x|/sqrt2)
  const float phi = (x >= 0.f) ? (1.0f - h) : h;
  return x * phi;
}

// Two elements at a time: the polynomial runs on the packed-fp32 pipe (FFMA2 on sm_100: one issue slot per pair), so the
// GELU epilogue of the MLP-up GEMM spends 6 + 2 x 5 instead of 2 x 11 FMA/ALU-pipe slots per pair.  Same arithmetic
// (round-to-nearest FMAs in the same order) as gelu_erf_fast: bit-identical results.
__device__ __forceinline__ uint64_t f32x2_pack(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ uint64_t f32x2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ void gelu_erf_fast2(float x0, float x1, float& y0, float& y1) {
  const float z0 = fminf(fabsf(x0) * 0.70710678118654752f, 4.3f);
  const float z1 = fminf(fabsf(x1) * 0.70710678118654752f, 4.3f);
  const uint64_t z = f32x2_pack(z0, z1);
  uint64_t q = f32x2_pack(2.699725252e-04f, 2.699725252e-04f);
  q = f32x2_fma(q, z, f32x2_pack(-4.347565948e-03f, -4.347565948e-03f));
  q = f32x2_fma(q, z, f32x2_pack(3.221176717e-02f, 3.221176717e-02f));
  q = f32x2_fma(q, z, f32x2_pack(-1.508187237e-01f, -1.508187237e-01f));
  q = f32x2_fma(q, z, f32x2_pack(-9.177533792e-01f, -9.177533792e-01f));
  q = f32x2_fma(q, z, f32x2_pack(-1.627978526e+00f, -1.627978526e+00f));
  q = f32x2_fma(q, z, f32x2_pack(-9.999988147e-01f, -9.999988147e-01f));
  float q0, q1, h0, h1;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(q0), "=f"(q1) : "l"(q));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(h0) : "f"(q0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(h1) : "f"(q1));
  y0 = x0 * ((x0 >= 0.f) ? (1.0f - h0) : h0);
  y1 = x1 * ((x1 >= 0.f) ? (1.0f - h1) : h1);
}

// "Residual from the pre-LayerNorm sums" (GemmArgs::resid_y): per tile, the source rows and LayerNorm statistics of the
// eight rows this lane adds residuals to (rows (lane >> 3) + 4 i of the warp's 32-row slab, the coalesced store
// layout).  Loaded BEFORE the wait for the accumulator, so neither the row-map -> sums dependency nor the statistics
// sit in the per-chunk critical path (loaded per chunk, the two dependent round trips made the residual GEMMs 40 %
// slower than with (hi, lo) pairs).
struct GemmResidRows {
  int src[8];
  float2 ms[8];      // (mean, rstd)
};
template <int EPI, bool SPLIT>
__device__ __forceinline__ void gemm_resid_rows(const GemmArgs& args, int M, int m0, int quarter, int lane, GemmResidRows& rr) {
  if constexpr (EPI == EPI_RESID_F32 && !SPLIT) {
    if (args.resid_y) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        // rows past M read row 0 (valid memory, result unused): every load below is unconditional, so the compiler
        // issues the eight of a chunk back to back (as branches they were serialised: one exposed latency each)
        const int grow = min(m0 + quarter * 32 + (lane >> 3) + 4 * i, M - 1);
        rr.src[i] = args.resid_src ? __ldg(args.resid_src + grow) : grow;
        rr.ms[i] = __ldg(args.resid_stats + grow);
      }
    }
  }
}

// Epilogue of one 128-row x BLOCK_N accumulator for one epilogue warp (TMEM lane quarter `quarter`, column half
// `half` of PARTS column parts): TMEM -> registers -> (+bias, activation) -> per-warp swizzled smem transpose -> coalesced global stores.
template <int BLOCK_N, int EPI, int PARTS = 2, bool SPLIT = false>
__device__ __forceinline__ void gemm_epilogue_warp(const GemmArgs& args, int M, int m0, int n0, uint32_t tmem_acc,
                                                   uint8_t* stg, int quarter, int half, int lane, const GemmResidRows& rr) {
      const int row_base = m0 + quarter * 32;     // first row of this warp's 32-row slab
      const int row = row_base + lane;
      const bool row_ok = row < M;
      int v_slot = 0, v_tok = 0;                  // EPI_QKV: the (slot, token) this thread's row belongs to
      if constexpr (EPI == EPI_QKV) {
        if (row_ok && n0 + BLOCK_N > args.qk_cols) {          // this tile holds V columns
          // proportional guess (exact for equal-length documents), then walk: row0[s] <= row < row0[s + 1]
          const int ns = *args.n_slots_dev;
          int sl = static_cast<int>(static_cast<float>(row) * (static_cast<float>(ns) / static_cast<float>(M)));   // a guess: float is fine
          sl = max(min(sl, ns - 1), 0);
          while (__ldg(args.row0 + sl) > row) --sl;
          while (__ldg(args.row0 + sl + 1) <= row) ++sl;
          v_slot = sl;
          v_tok = row - __ldg(args.row0 + sl);
        }
      }
      const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(quarter * 32) << 16);

#pragma unroll 1
      for (int c = half * (BLOCK_N / PARTS); c < (half + 1) * (BLOCK_N / PARTS); c += 32) {
        const int n = n0 + c;
        uint2 rs[8], rl[8];
        float4 ln_g = make_float4(0.f, 0.f, 0.f, 0.f), ln_b = ln_g;   // resid_y: LayerNorm weight / bias of this lane's 4 columns
        if constexpr (EPI == EPI_RESID_F32 && !SPLIT) {
          if (args.resid_y) {
            ln_g = __ldg(reinterpret_cast<const float4*>(args.resid_w + n + (lane & 7) * 4));
            ln_b = __ldg(reinterpret_cast<const float4*>(args.resid_b + n + (lane & 7) * 4));
          }
        }
        if constexpr (EPI == EPI_RESID_F32) {       // residual loads first: independent of the accumulator
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int grow = row_base + (lane >> 3) + 4 * i;
            const size_t off = static_cast<size_t>(grow) * args.N + n + (lane & 7) * 4;
            if (SPLIT && args.resid_f32) {          // (rs, rl) hold the four fp32 residuals of this lane's 16 B
              const float4 r4 = (grow < M) ? __ldg(reinterpret_cast<const float4*>(args.resid_f32 + off)) : make_float4(0.f, 0.f, 0.f, 0.f);
              rs[i] = make_uint2(__float_as_uint(r4.x), __float_as_uint(r4.y));
              rl[i] = make_uint2(__float_as_uint(r4.z), __float_as_uint(r4.w));
            } else if (!SPLIT && args.resid_y) {    // the four fp32 pre-LayerNorm sums behind this lane's 16 B
              const float4 r4 = __ldg(reinterpret_cast<const float4*>(args.resid_y + static_cast<size_t>(rr.src[i]) * args.N + n + (lane & 7) * 4));
              rs[i] = make_uint2(__float_as_uint(r4.x), __float_as_uint(r4.y));
              rl[i] = make_uint2(__float_as_uint(r4.z), __float_as_uint(r4.w));
            } else {
              rs[i] = (grow < M) ? __ldg(reinterpret_cast<const uint2*>(args.resid + off)) : make_uint2(0u, 0u);
              rl[i] = (grow < M && args.resid_lo) ? __ldg(reinterpret_cast<const uint2*>(args.resid_lo + off)) : make_uint2(0u, 0u);
            }
          }
        }
        uint32_t v[32];
        tmem_ld32(taddr + c, v);
        uint64_t bv[16];                            // bias pairs for the packed-fp32 add (FADD2)
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 b4 = __ldg(reinterpret_cast<const float4*>(args.bias + n) + q);
          bv[q * 2 + 0] = f32x2_pack(b4.x, b4.y); bv[q * 2 + 1] = f32x2_pack(b4.z, b4.w);
        }
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          uint64_t x, y;
          asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "r"(v[2 * j]), "r"(v[2 * j + 1]));
          asm("add.rn.f32x2 %0, %1, %2;" : "=l"(y) : "l"(x), "l"(bv[j]));
          asm("mov.b64 {%0, %1}, %2;" : "=f"(f[2 * j]), "=f"(f[2 * j + 1]) : "l"(y));
        }

        if constexpr (EPI == EPI_BIAS_BF16 || EPI == EPI_GELU_BF16 || EPI == EPI_QKV) {
          bool transposed_v = false;
          if constexpr (EPI == EPI_QKV) transposed_v = (n >= args.qk_cols);
          if (!transposed_v) {
            if constexpr (EPI == EPI_GELU_BF16) {
#pragma unroll
              for (int j = 0; j < 32; j += 2) gelu_erf_fast2(f[j], f[j + 1], f[j], f[j + 1]);
            }
            // bf16 row slab: 64 B per row; thread = row writes 4 x 16 B chunks (chunk ^ ((row>>1)&3): conflict-free)
            // SPLIT: a second pass moves the low parts f - bf16(f) the same way
#pragma unroll
            for (int part = 0; part < (SPLIT ? 2 : 1); ++part) {
              __syncwarp();
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                uint32_t w[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const uint32_t hi = pack_bf16x2(f[q * 8 + 2 * j], f[q * 8 + 2 * j + 1]);
                  if (part == 0) {
                    w[j] = hi;
                  } else {
                    const float2 hf = unpack_bf16x2(hi);
                    w[j] = pack_bf16x2(f[q * 8 + 2 * j] - hf.x, f[q * 8 + 2 * j + 1] - hf.y);
                  }
                }
                *reinterpret_cast<uint4*>(stg + lane * 64 + ((q ^ ((lane >> 1) & 3)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
              }
              __syncwarp();
              // 4 lanes cover one row's 64 B; 8 rows per store instruction
              __nv_bfloat16* outp = part == 0 ? static_cast<__nv_bfloat16*>(args.out) : args.out_lo;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int r = (lane >> 2) + 8 * i, q = lane & 3;
                const uint4 val = *reinterpret_cast<const uint4*>(stg + r * 64 + ((q ^ ((r >> 1) & 3)) << 4));
                if (row_base + r < M)
                  *reinterpret_cast<uint4*>(outp + static_cast<size_t>(row_base + r) * args.ld_out + n + q * 8) = val;
              }
            }
          } else if (row_ok) {
            // V is stored transposed per (doc, head): vt[d][token] so that P*V takes a K-major B operand.
            const int doc = v_slot, tok = v_tok;
            const int nv = n - args.qk_cols;        // 32-aligned => one head per chunk
            const int head = nv >> 6;
            const int d0 = nv & 63;
            const size_t voff = (static_cast<size_t>(doc * args.heads + head) * 64 + d0) * args.kv_pitch + tok;
            __nv_bfloat16* dst = args.vt + voff;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const __nv_bfloat16 hi = __float2bfloat16_rn(f[j]);
              dst[static_cast<size_t>(j) * args.kv_pitch] = hi;
              if constexpr (SPLIT)
                args.vt_lo[voff + static_cast<size_t>(j) * args.kv_pitch] = __float2bfloat16_rn(f[j] - __bfloat162float(hi));
            }
          }
        } else {
          // fp32 row slab: 128 B per row; thread = row writes 8 x 16 B chunks (chunk ^ (row&7): conflict-free)
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(stg + lane * 128 + ((q ^ (lane & 7)) << 4)) =
                make_float4(f[q * 4 + 0], f[q * 4 + 1], f[q * 4 + 2], f[q * 4 + 3]);
          __syncwarp();
          // 8 lanes cover one row's 128 B; 4 rows per store instruction; residual / pos-embed added here (coalesced)
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = (lane >> 3) + 4 * i, q = lane & 7;
            float4 val = *reinterpret_cast<const float4*>(stg + r * 128 + ((q ^ (r & 7)) << 4));
            const int grow = row_base + r;
            if (grow < M) {
              if constexpr (EPI == EPI_RESID_F32) {
                if (SPLIT && args.resid_f32) {
                  val.x += __uint_as_float(rs[i].x); val.y += __uint_as_float(rs[i].y);
                  val.z += __uint_as_float(rl[i].x); val.w += __uint_as_float(rl[i].y);
                } else if (!SPLIT && args.resid_y) {
                  // the LayerNorm kernel's own expression (ln_rows_vec_kernel), on the sums it read
                  const float2 ms = rr.ms[i];       // q == lane & 7: ln_g / ln_b are this lane's columns
                  val.x += (__uint_as_float(rs[i].x) - ms.x) * ms.y * ln_g.x + ln_b.x;
                  val.y += (__uint_as_float(rs[i].y) - ms.x) * ms.y * ln_g.y + ln_b.y;
                  val.z += (__uint_as_float(rl[i].x) - ms.x) * ms.y * ln_g.z + ln_b.z;
                  val.w += (__uint_as_float(rl[i].y) - ms.x) * ms.y * ln_g.w + ln_b.w;
                } else {
                  const float2 r0 = unpack_bf16x2(rs[i].x), r1 = unpack_bf16x2(rs[i].y);
                  const float2 l0 = unpack_bf16x2(rl[i].x), l1 = unpack_bf16x2(rl[i].y);
                  val.x += r0.x + l0.x; val.y += r0.y + l0.y; val.z += r1.x + l1.x; val.w += r1.y + l1.y;
                }
                *reinterpret_cast<float4*>(static_cast<float*>(args.out) + static_cast<size_t>(grow) * args.ld_out + n + q * 4) = val;
              } else {   // EPI_PATCH
                const int doc = grow / args.n_patch;
                const int p = grow - doc * args.n_patch;
                const float4 pe = __ldg(reinterpret_cast<const float4*>(args.pos + static_cast<size_t>(1 + p) * args.N + n + q * 4));
                val.x += pe.x; val.y += pe.y; val.z += pe.z; val.w += pe.w;
                *reinterpret_cast<float4*>(static_cast<float*>(args.out) +
                    (static_cast<size_t>(doc) * args.n_vis + 1 + p) * args.ld_out + n + q * 4) = val;
              }
            }
          }
        }
      }
}

template <int BLOCK_N, int EPI, bool SPLIT = false>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_a_lo, const __grid_constant__ CUtensorMap tmap_b_lo,
               const GemmArgs args) {
  using SM = GemmSmem<BLOCK_N>;
  constexpr int STAGES = SM::STAGES;
  constexpr uint32_t TMEM_COLS = (2 * BLOCK_N <= 256) ? 256 : 512;

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + SM::BAR_OFF);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int M = args.m_dev ? *args.m_dev : args.m_static;
  if (M <= 0) return;              // every document has left: no barrier / TMEM set-up for an empty launch
  const int m_blocks = (M + GEMM_BLOCK_M - 1) / GEMM_BLOCK_M;
  const int n_blocks = args.N / BLOCK_N;
  const int k_blocks = args.K / GEMM_BLOCK_K;
  const int k_iters = SPLIT ? 3 * k_blocks : k_blocks;       // SPLIT: A_hi W_hi, A_lo W_hi, A_hi W_lo over the same k range
  const int total_tiles = m_blocks * n_blocks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if constexpr (SPLIT) { tma_prefetch_desc(&tmap_a_lo); tma_prefetch_desc(&tmap_b_lo); }
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], GEMM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<TMEM_COLS>(tmem_base_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_blocks) * GEMM_BLOCK_M;
        const int n0 = (tile % n_blocks) * BLOCK_N;
        for (int it = 0; it < k_iters; ++it) {
          const int seg = SPLIT ? it / k_blocks : 0, kb = it - seg * k_blocks;
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * SM::STAGE_BYTES;
          uint8_t* sb = sa + SM::A_BYTES;
          mbar_expect_tx(&full_bar[stage], SM::STAGE_BYTES);
          tma_load_2d(sa, seg == 1 ? &tmap_a_lo : &tmap_a, &full_bar[stage], kb * GEMM_BLOCK_K, m0);
          tma_load_2d(sb, seg == 2 ? &tmap_b_lo : &tmap_b, &full_bar[stage], kb * GEMM_BLOCK_K, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(GEMM_BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < k_iters; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * SM::STAGE_BYTES);
          const uint32_t sb = sa + SM::A_BYTES;
          const uint64_t da = umma_desc_sw128_kmajor(sa);
          const uint64_t db = umma_desc_sw128_kmajor(sb);
#pragma unroll
          for (int k = 0; k < GEMM_BLOCK_K / 16; ++k) {
            // +32 B per K=16 step inside the 128 B swizzle row (descriptor address is in 16 B units)
            umma_bf16_ss(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tmem_full[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (2..9)
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;             // which half of the tile's columns
    uint8_t* stg = smem + SM::STG_OFF + (warp - 2) * 4096;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int m0 = (tile / n_blocks) * GEMM_BLOCK_M;
      const int n0 = (tile % n_blocks) * BLOCK_N;
      if constexpr (EPI == EPI_RESID_F32) {
        // pull the NEXT tile's residual slab (32 rows x BLOCK_N/2 bf16 of this warp) into L2 while this tile's
        // MMAs are still running: the residual was written a layer ago and has long left the cache
        const int nt = tile + gridDim.x;
        if (nt < total_tiles && args.resid) {
          const int pr = (nt / n_blocks) * GEMM_BLOCK_M + quarter * 32 + lane;
          if (pr < M) {
            const __nv_bfloat16* pp = args.resid + static_cast<size_t>(pr) * args.N + (nt % n_blocks) * BLOCK_N +
                                      half * (BLOCK_N / 2);
#pragma unroll
            for (int b = 0; b < BLOCK_N; b += 128)      // BLOCK_N/2 bf16 = BLOCK_N bytes per row
              asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(pp) + b));
          }
        }
      }
      GemmResidRows rr;
      gemm_resid_rows<EPI, SPLIT>(args, M, m0, quarter, lane, rr);
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      gemm_epilogue_warp<BLOCK_N, EPI, 2, SPLIT>(args, M, m0, n0, tmem_base + acc * BLOCK_N, stg, quarter, half, lane, rr);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2): a cluster of two CTAs on one TPC computes a 256 x 256 tile.  Each CTA stages
// its own 128 rows of A and HALF of the weight tile (128 of the 256 output columns); the pair's tensor cores read
// both halves, so every k-block moves 32 KB per SM through L2 instead of 48 KB (the single-CTA kernel is bound by
// L2 -> SM operand traffic at these shapes, see profiles/).  The leader (cluster rank 0) issues every MMA; its
// tcgen05.commit is multicast to the stage / accumulator barriers of both CTAs; both CTAs' epilogue warps release
// the accumulator on the leader's barrier.  Epilogue as above, each CTA for its own 128 rows.
// EPI_WARPS: 8 (two column halves per TMEM lane quarter) or 16 (four column quarters: twice the epilogue issue
// bandwidth for the math-heavy GELU / QKV epilogues; the residual epilogue needs too many registers for 576 threads).
template <int EPI_WARPS>
struct GemmPairSmemT {
  static constexpr int STAGES = 5;
  static constexpr int A_BYTES = GEMM_BLOCK_M * GEMM_BLOCK_K * 2;       // 16 KB
  static constexpr int B_BYTES = 128 * GEMM_BLOCK_K * 2;                // 16 KB: this CTA's half of the 256 columns
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STG_OFF = STAGES * STAGE_BYTES;
  static constexpr int BAR_OFF = STG_OFF + EPI_WARPS * 4096;
  static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 4) * 8 + 16;
  static constexpr int DYN_BYTES = TOTAL;                               // dynamic smem base is 1024 B aligned
  static constexpr int THREADS = 64 + EPI_WARPS * 32;
};
using GemmPairSmem = GemmPairSmemT<8>;
template <int EPI>
__host__ __device__ constexpr int gemm_pair_epi_warps() { return EPI == EPI_RESID_F32 ? 8 : 16; }

template <int EPI, bool SPLIT = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + gemm_pair_epi_warps<EPI>() * 32, 1)
gemm_tc_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const __grid_constant__ CUtensorMap tmap_a_lo, const __grid_constant__ CUtensorMap tmap_b_lo,
                    const GemmArgs args) {
  constexpr int EPI_WARPS = gemm_pair_epi_warps<EPI>();
  constexpr int PARTS = EPI_WARPS / 4;
  using SM = GemmPairSmemT<EPI_WARPS>;
  constexpr int STAGES = SM::STAGES;
  constexpr int BLOCK_N = 256;
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t sb = smem_u32(smem);
  if (sb & 1023u) __trap();
  const uint32_t full_bar = sb + SM::BAR_OFF;                  // [STAGES]  (used in the leader only)
  const uint32_t empty_bar = full_bar + STAGES * 8;            // [STAGES]  local to each CTA
  const uint32_t tmem_full = empty_bar + STAGES * 8;           // [2]       local to each CTA
  const uint32_t tmem_empty = tmem_full + 2 * 8;               // [2]       (used in the leader only)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM::BAR_OFF);
  uint32_t* tmem_base_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;

  const int M = args.m_dev ? *args.m_dev : args.m_static;
  if (M <= 0) return;              // every document has left (both CTAs of the pair read the same M): empty launch
  const int m_blocks = (M + 2 * GEMM_BLOCK_M - 1) / (2 * GEMM_BLOCK_M);      // 256-row tiles
  const int n_blocks = args.N / BLOCK_N;
  const int k_blocks = args.K / GEMM_BLOCK_K;
  const int k_iters = SPLIT ? 3 * k_blocks : k_blocks;       // SPLIT: A_hi W_hi, A_lo W_hi, A_hi W_lo over the same k range
  const int total_tiles = m_blocks * n_blocks;
  const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    if constexpr (SPLIT) { tma_prefetch_desc(&tmap_a_lo); tma_prefetch_desc(&tmap_b_lo); }
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(bars + i, 1);                       // full: the leader's expect_tx arrival
      mbar_init(bars + STAGES + i, 1);              // empty: multicast commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bars + 2 * STAGES + i, 1);                          // tmem_full: multicast commit
      mbar_init(bars + 2 * STAGES + 2 + i, 2 * EPI_WARPS);          // tmem_empty: epilogue warps of both CTAs
    }
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc_pair<512>(tmem_base_slot);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_base_slot;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = pair; tile < total_tiles; tile += n_pairs) {
        const int m0 = (tile / n_blocks) * 2 * GEMM_BLOCK_M + static_cast<int>(rank) * GEMM_BLOCK_M;
        const int n0 = (tile % n_blocks) * BLOCK_N + static_cast<int>(rank) * (BLOCK_N / 2);
        for (int it = 0; it < k_iters; ++it) {
          const int seg = SPLIT ? it / k_blocks : 0, kb = it - seg * k_blocks;
          mbar_wait(empty_bar + stage * 8, phase ^ 1);
          const uint32_t sa = sb + stage * SM::STAGE_BYTES;
          if (leader) mbar_expect_tx(full_bar + stage * 8, 2 * SM::STAGE_BYTES);   // both CTAs' bytes land on it
          tma_load_2d_pair(sa, seg == 1 ? &tmap_a_lo : &tmap_a, full_bar + stage * 8, kb * GEMM_BLOCK_K, m0);
          tma_load_2d_pair(sa + SM::A_BYTES, seg == 2 ? &tmap_b_lo : &tmap_b, full_bar + stage * 8, kb * GEMM_BLOCK_K, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA only)
    if (leader && elect_one()) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * GEMM_BLOCK_M, BLOCK_N);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = pair; tile < total_tiles; tile += n_pairs) {
        mbar_wait(tmem_empty + acc * 8, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
        for (int kb = 0; kb < k_iters; ++kb) {
          mbar_wait(full_bar + stage * 8, phase);
          tc_fence_after();
          const uint32_t sa = sb + stage * SM::STAGE_BYTES;
          const uint64_t da = umma_desc_sw128_kmajor(sa);
          const uint64_t db = umma_desc_sw128_kmajor(sa + SM::A_BYTES);
#pragma unroll
          for (int k = 0; k < GEMM_BLOCK_K / 16; ++k)
            umma_bf16_ss_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          umma_commit_pair(empty_bar + stage * 8);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(tmem_full + acc * 8);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps (2..), both CTAs
    const int quarter = warp & 3;
    const int half = (warp - 2) >> 2;
    uint8_t* stg = smem + SM::STG_OFF + (warp - 2) * 4096;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = pair; tile < total_tiles; tile += n_pairs) {
      const int m0 = (tile / n_blocks) * 2 * GEMM_BLOCK_M + static_cast<int>(rank) * GEMM_BLOCK_M;
      const int n0 = (tile % n_blocks) * BLOCK_N;
      if constexpr (EPI == EPI_RESID_F32 && !SPLIT) {
        // the residual sums of the NEXT tile of this pair (this lane's row, this warp's column part: BLOCK_N / PARTS
        // fp32) -> L2: they were written a GEMM or a layer ago and have long left the cache
        const int nt = tile + n_pairs;
        if (args.resid_y && args.resid_prefetch && nt < total_tiles) {
          const int pr = (nt / n_blocks) * 2 * GEMM_BLOCK_M + static_cast<int>(rank) * GEMM_BLOCK_M + quarter * 32 + lane;
          if (pr < M) {
            const size_t srow = args.resid_src ? static_cast<size_t>(__ldg(args.resid_src + pr)) : static_cast<size_t>(pr);
            const char* pp = reinterpret_cast<const char*>(args.resid_y + srow * args.N + (nt % n_blocks) * BLOCK_N +
                                                           half * (BLOCK_N / PARTS));
#pragma unroll
            for (int b = 0; b < (BLOCK_N / PARTS) * 4; b += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(pp + b));
          }
        }
      }
      GemmResidRows rr;
      gemm_resid_rows<EPI, SPLIT>(args, M, m0, quarter, lane, rr);
      mbar_wait(tmem_full + acc * 8, acc_phase);
      tc_fence_after();
      gemm_epilogue_warp<BLOCK_N, EPI, PARTS, SPLIT>(args, M, m0, n0, tmem_base + acc * BLOCK_N, stg, quarter, half, lane, rr);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tmem_empty + acc * 8, 0);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair<512>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side: shapes, tensor maps, launch
// The engine and the GEMM tests (tests/kernels/gemm_harness.cu) both launch through these, so the tests run the
// engine's own launch.

// BLOCK_N of a GEMM with N = n output columns: 256 (the CTA-pair kernel) when it divides n, else 128.
inline int gemm_block_n(int n) { return (n % 256 == 0) ? 256 : 128; }

// BLOCK_N of the QKV GEMM (N = 3H): a tile holds either Q|K or V^T columns, so 2H must be a multiple of it.
inline int gemm_block_n_qkv(int H) {
  const int bn = gemm_block_n(H);
  return (2 * H) % bn ? 128 : bn;
}

// fp32 engine mode: the tensor core adds each K = 16 product block into the fp32 accumulator with truncation, so the
// error of a long contraction grows linearly with K.  The MLP-down GEMM (K = I) therefore runs in K chunks of this many
// columns, each its own launch whose residual epilogue adds the running sum in fp32 (round to nearest).
inline int gemm_kchunk(int I) { return (I > 1024 && I % 1024 == 0) ? 1024 : ((I > 768 && I % 768 == 0) ? 768 : I); }

// Weight TMA box rows: each CTA of a pair (BLOCK_N = 256) stages half of the 256 output columns.
inline int gemm_wbox(int bn) { return bn == 256 ? 128 : bn; }

// A operand: columns [col0, col0 + K) of `rows` bf16 rows at row pitch `pitch` (col0 > 0: a K chunk).
inline CUtensorMap gemm_a_map(const __nv_bfloat16* a, uint64_t rows, uint64_t K, uint64_t pitch, size_t col0 = 0) {
  return make_tmap_2d_sw128(a + col0, rows, K, pitch, GEMM_BLOCK_M);
}

// Weight [N, K] of a GEMM family with BLOCK_N = bn: columns [col0, col0 + K) of bf16 rows at row pitch `pitch`.
inline CUtensorMap gemm_w_map(const __nv_bfloat16* w, uint64_t N, uint64_t K, uint64_t pitch, int bn, size_t col0 = 0) {
  return make_tmap_2d_sw128(w + col0, N, K, pitch, gemm_wbox(bn));
}

// static (internal linkage) here and below: every library built from this header (the engine, a test harness) keeps its
// own attribute cache for its own copy of the kernels.  A static of an inline function would be one object per process.
template <int EPI, bool SPLIT>
static void launch_gemm_kernel(int device, int sms, int bn, const CUtensorMap& ta, const CUtensorMap& tb,
                               const CUtensorMap& ta_lo, const CUtensorMap& tb_lo, const GemmArgs& a, cudaStream_t st,
                               int grid) {
  // the shared-memory attribute is per device; it is set by the first launch, before a plan captures a forward
  if (bn == 256) {
    using PS = GemmPairSmemT<gemm_pair_epi_warps<EPI>()>;
    static bool configured[64] = {};
    if (!configured[device & 63]) {
      CUDA_OK(cudaFuncSetAttribute(gemm_tc_pair_kernel<EPI, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   PS::DYN_BYTES));
      configured[device & 63] = true;
    }
    gemm_tc_pair_kernel<EPI, SPLIT><<<grid ? grid : (sms & ~1), PS::THREADS, PS::DYN_BYTES, st>>>(ta, tb, ta_lo, tb_lo, a);
  } else {
    static bool configured[64] = {};
    if (!configured[device & 63]) {
      CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<128, EPI, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   GemmSmem<128>::DYN_BYTES));
      configured[device & 63] = true;
    }
    gemm_tc_kernel<128, EPI, SPLIT><<<grid ? grid : sms, GEMM_THREADS, GemmSmem<128>::DYN_BYTES, st>>>(ta, tb, ta_lo, tb_lo, a);
  }
  CUDA_OK(cudaGetLastError());
}

// One GEMM on `device` (an ordinal, passed in so a launch queries nothing) with `sms` SMs.  bn: 128 (gemm_tc_kernel)
// or 256 (gemm_tc_pair_kernel, CTA pairs).  split (fp32 engine mode): ta_lo / tb_lo are the low parts' maps; in bf16
// mode they are ignored.  grid 0: one CTA per SM (pairs: an even count); another grid gives the same result.
template <int EPI>
static void launch_gemm(int device, int sms, int bn, bool split, const CUtensorMap& ta, const CUtensorMap& tb,
                        const CUtensorMap& ta_lo, const CUtensorMap& tb_lo, const GemmArgs& a, cudaStream_t st, int grid = 0) {
  if (split) launch_gemm_kernel<EPI, true>(device, sms, bn, ta, tb, ta_lo, tb_lo, a, st, grid);
  else launch_gemm_kernel<EPI, false>(device, sms, bn, ta, tb, ta, tb, a, st, grid);
}

}  // namespace mmee
