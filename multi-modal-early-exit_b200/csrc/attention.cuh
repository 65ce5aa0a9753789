// Fused attention for LayoutLMv3 (HF modeling_layoutlmv3.py:236-289):
//     ctx = softmax( (Q/8) K^T + (rel_pos + rel_2d_pos)/8 + key_mask ) V
// Persistent kernel, TWO co-resident CTAs per SM (grid = 2 x #SMs), work item = (document slot, head,
// 128-query tile), 64-key tiles.  Everything between Q/K/V and ctx stays on the SM:
//   S_t  = Q K_t^T + B_t I    tcgen05.mma 128x64x64 twice into the same fp32 TMEM accumulator: bf16 Q.K^T (Q resident in
//                             TMEM for the whole item, copied there once by the softmax warps), then the
//                             fp16 bias tile B_t (relative-position bias in the log2 domain with -60000 on padded
//                             keys, built once per forward by bias_build_kernel, streamed by TMA) times a 64x64
//                             identity -- the bias add and the key mask cost no thread instruction
//   P_t  = exp2(S_t - ref)    one softmax thread per query row (= TMEM lane): tcgen05.ld, FADD, MUFU.EX2, bf16 pairs
//                             written back INTO the S buffer with tcgen05.st
//   O   += P_t [V_t | 1]      tcgen05.mma 128x80x64 with the A operand (P) read from TMEM (TS form); O (64 dims +
//                             the row sum of P from a ones-row appended to V^T) accumulates in TMEM over the item
// so neither the [S,S] scores nor P ever touch shared or global memory, and O is read back once per item.
// The CogView "PB-relax" softmax of HF:224-234 is the standard max-shifted softmax.  Fully padded key tiles are
// skipped (slot_meta).
//
// Roles per CTA (192 threads): warp 0 TMA producer, warp 1 MMA issuer (+TMEM owner), warps 2-5 softmax.
// S_{t+1} is issued before P V_t, and P V_t only needs P_t, so the softmax warps never wait on the tensor core in
// steady state; the two CTAs of an SM fill each other's MUFU bubbles.
//
// Everything runs in the log2 domain (log2(e)/sqrt(d) is folded into W_q and into the bias).  The first tile of an
// item takes its exact row maximum as reference.  Later tiles keep it unless a score exceeds it by more than 2^8
// (lazy rescaling: P <= 256 is harmless in bf16/fp32); then the reference is raised for the following tiles and O
// is rescaled in place in TMEM by exp2(old - new) before the next P V.  A score more than 2^40 above the reference
// takes an exact path: the reference is raised at once, the row's P is recomputed and O rescaled before this P V.
#pragma once
#include <cuda.h>

#include <type_traits>

#include "ptx.cuh"
#include "tmap.h"

namespace mmee {

constexpr int ATT_SM_WARPS = 4;      // softmax warps: one thread per query row
constexpr int ATT_THREADS = 64 + ATT_SM_WARPS * 32;
constexpr int ATT_CTAS_PER_SM = 2;
constexpr int ATT_BQ = 128;    // query rows per CTA
constexpr int ATT_BKV = 64;    // keys per tile
constexpr int ATT_D = 64;
constexpr int ATT_DV = 80;     // V^T rows fed to the PV MMA: 64 dims + a ones row (row sum of P) + 15 zero rows
constexpr int ATT_KB_STAGES = 2;  // K + bias ring: a stage is released as soon as S_t = Q K^T + B I has been computed
constexpr int ATT_V_STAGES = 2;   // V^T ring: released when P V_t has completed
constexpr int ATT_MAX_KV_TILES = 16;
constexpr float ATT_LAZY = 8.0f;   // raise the row reference only when a score exceeds it by more than 2^8
constexpr float ATT_JUMP = 40.0f;  // ... and immediately (P recomputed) when it exceeds it by more than 2^40

// kSplit (fp32 engine mode): Q, K, V^T, the bias and P are split-bf16 / split-fp16 pairs (hi + lo); S, O and the
// softmax stay fp32, so each tile runs Q_hi K_hi + Q_lo K_hi + Q_hi K_lo (+ B_hi I + B_lo I) and
// P_hi [V_hi|1] + P_lo [V_hi|1] + P_hi V_lo.  One CTA per SM (twice the operand tiles, 512 TMEM columns).
template <bool kSplit>
struct AttSmemT {
  static constexpr int NP = kSplit ? 2 : 1;                    // operand parts
  static constexpr int Q_BYTES = ATT_BQ * ATT_D * 2;           // 16 KB per part
  static constexpr int K_BYTES = ATT_BKV * ATT_D * 2;          //  8 KB per part
  static constexpr int V_BYTES = ATT_DV * ATT_BKV * 2;         // 10 KB: [80 rows x 64 keys] bf16, SW128 (hi part, with the ones row)
  static constexpr int VLO_BYTES = kSplit ? ATT_D * ATT_BKV * 2 : 0;   //  8 KB: [64 rows x 64 keys] low part
  static constexpr int B_BYTES = ATT_BQ * ATT_BKV * 2;         // 16 KB  fp16 [128 x 64] per part, SW128 (A operand of the bias MMA)
  static constexpr int Q_STAGE = NP * Q_BYTES;
  static constexpr int KB_STAGE = NP * (K_BYTES + B_BYTES);    // 24 KB (48 KB split): K parts, then bias parts
  static constexpr int V_STAGE = V_BYTES + VLO_BYTES;
  static constexpr int I_BYTES = ATT_BKV * ATT_BKV * 2;        //  8 KB  fp16 identity [64 x 64], SW128 (B operand)
  static constexpr int Q_OFF = 0;                              // 2 Q buffers
  static constexpr int KB_OFF = Q_OFF + 2 * Q_STAGE;
  static constexpr int V_OFF = KB_OFF + ATT_KB_STAGES * KB_STAGE;
  static constexpr int I_OFF = V_OFF + ATT_V_STAGES * V_STAGE;
  static constexpr int BAR_OFF = I_OFF + I_BYTES;
  // q_full[2] q_empty[2] kb_full[KB] kb_empty[KB] v_full[V] v_empty[V] s_full[2] p_full[2] o_full[1] qt_full[1]
  static constexpr int N_BARS = 2 + 2 + 2 * ATT_KB_STAGES + 2 * ATT_V_STAGES + 2 + 2 + 1 + 1;
  static constexpr int TOTAL = BAR_OFF + N_BARS * 8 + 16;
  static constexpr int DYN_BYTES = TOTAL;                      // the dynamic smem base itself is 1024 B aligned
  static constexpr uint32_t TMEM_COLS = kSplit ? 512 : 256;
};
using AttSmem = AttSmemT<false>;
static_assert(AttSmem::DYN_BYTES <= 115712, "two attention CTAs must fit one SM");
static_assert(AttSmemT<true>::DYN_BYTES <= 232448, "split attention CTA must fit one SM");
static_assert(AttSmem::KB_STAGE % 1024 == 0 && AttSmem::K_BYTES % 1024 == 0 && AttSmem::V_BYTES % 1024 == 0 &&
                  AttSmem::V_OFF % 1024 == 0 && AttSmem::I_OFF % 1024 == 0 && AttSmemT<true>::V_STAGE % 1024 == 0 &&
                  AttSmemT<true>::V_OFF % 1024 == 0 && AttSmemT<true>::I_OFF % 1024 == 0,
              "swizzled tiles need 1024 B alignment");

struct AttArgs {
  // ragged work list of the exit stage (norm_exit.cuh SlotRows, written by plan_rows_block): slot s owns rows
  // [meta[s].x, meta[s].x + meta[s].y) of Q / K / ctx, belongs to document meta[s].z and its query tiles are numbers
  // meta[s].w ... in qt_slot; item = heads * meta[s].w + head * n_qt(s) + query tile
  const int4* slot_meta;
  const int* qt_slot;
  const int* n_qt_dev;
  int* err_flag;               // guard: set to 1 if a deferred rescale factor underflowed (unreachable, see ATT_JUMP)
  long long* trace;            // developer trace (kTrace instantiation only): clock64 stamps of CTA 0
  __nv_bfloat16* ctx;          // [M, H]
  __nv_bfloat16* ctx_lo;       // kSplit: low part of ctx
  int H, heads, seq;           // seq: token pitch of the bias rows (max tokens per document)
  int tail16;                  // a last key tile with <= 16 real keys runs as a 16-key tile
  int experiment;              // developer timing experiment (results are WRONG): bit 0 skip K / V^T loads, bit 1 skip bias loads
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// (a, b) + (c, c) as one packed-fp32 add (FADD2 on sm_100): half the issue slots of two FADDs
__device__ __forceinline__ void sub_ref_x2(uint32_t a, uint32_t b, uint64_t nref2, float& ya, float& yb) {
  uint64_t x, y;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "r"(a), "r"(b));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(y) : "l"(x), "l"(nref2));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(ya), "=f"(yb) : "l"(y));
}

// Position in this CTA's (item, key tile) sequence.  Every role walks the same sequence so the pipeline counters stay
// in lock-step.  Passed by value so it lives in registers.  An item = (slot, head, 128-row query tile); its key tiles
// are 0 .. last_j (documents are ragged: only kept tokens have rows, so there are no padded key tiles to skip).
struct AttCursor {
  int item, ii, j, slot, head, q0, doc, last_j, tail_j, row0, rows;
  int nitem;                   // the NEXT item this CTA processes (>= total_items: none)
  int4 nmeta;                  // its slot meta, loaded one item ahead (latency hidden)
  bool valid;
};

__device__ __forceinline__ int4 att_item_meta(int item, int total_items, const AttArgs& args) {
  return (item < total_items) ? __ldg(args.slot_meta + __ldg(args.qt_slot + item / args.heads)) : make_int4(0, 1, 0, 0);
}
__device__ __forceinline__ AttCursor att_enter(int item, int ii, int4 meta, int total_items, int stride,
                                               const AttArgs& args) {
  AttCursor c;
  c.item = item; c.ii = ii; c.valid = item < total_items;
  c.j = 0; c.slot = 0; c.head = 0; c.q0 = 0; c.doc = 0; c.last_j = 0; c.tail_j = -1; c.row0 = 0; c.rows = 1;
  c.nmeta = make_int4(0, 1, 0, 0);
  c.nitem = total_items;
  if (!c.valid) return c;
  c.row0 = meta.x; c.rows = meta.y; c.doc = meta.z;
  const int n_qt = (c.rows + ATT_BQ - 1) / ATT_BQ;
  const int local = item - args.heads * meta.w;
  c.head = local / n_qt;
  c.q0 = (local - c.head * n_qt) * ATT_BQ;
  c.slot = __ldg(args.qt_slot + item / args.heads);
  c.last_j = (c.rows + ATT_BKV - 1) / ATT_BKV - 1;
  const int rem = c.rows - c.last_j * ATT_BKV;           // real keys of the last tile
  c.tail_j = (args.tail16 && c.last_j > 0 && rem <= 16) ? c.last_j : -1;
  c.nitem = item + stride;
  c.nmeta = att_item_meta(c.nitem, total_items, args);
  return c;
}
__device__ __forceinline__ AttCursor att_first(int total_items, int stride, const AttArgs& args) {
  const int item = blockIdx.x;
  return att_enter(item, 0, att_item_meta(item, total_items, args), total_items, stride, args);
}
__device__ __forceinline__ AttCursor att_next(AttCursor c, int total_items, int stride, const AttArgs& args) {
  if (c.j < c.last_j) { ++c.j; return c; }
  return att_enter(c.nitem, c.ii + 1, c.nmeta, total_items, stride, args);
}

// tmap_q   : bf16 [M_max, 2H]                    box [128 rows x 64 cols]   (SW128)
// tmap_k   : bf16 [M_max, 2H]                    box [ 64 rows x 64 cols]   (SW128)
// tmap_vt  : bf16 [docs*heads*64, kv_pitch]       box [ 64 rows x 64 cols]   (SW128)
// tmap_bias: fp16 [docs*heads*seq, bias_pitch]    box [128 rows x 64 cols]   (SW128)
// kSplit: the *_lo maps describe the low parts (same shapes); otherwise they are unused copies
struct AttMaps {
  CUtensorMap q, k, vt, bias, q_lo, k_lo, vt_lo, bias_lo;
};

template <bool kTrace, bool kSplit = false>
__global__ void __launch_bounds__(ATT_THREADS, kSplit ? 1 : ATT_CTAS_PER_SM)
attention_kernel(const __grid_constant__ AttMaps maps, const AttArgs args) {
  using SMEM = AttSmemT<kSplit>;
  const CUtensorMap& tmap_q = maps.q;
  const CUtensorMap& tmap_k = maps.k;
  const CUtensorMap& tmap_vt = maps.vt;
  const CUtensorMap& tmap_bias = maps.bias;
  const int S = args.seq;
  const int total_items = *args.n_qt_dev * args.heads;
  const int stride = gridDim.x;
  if (total_items == 0) return;    // every document has left: no barrier / TMEM set-up for an empty launch

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 32-bit shared-window address of the working area; all hot-loop accesses use these addresses
  const uint32_t sb = smem_u32(smem_raw);
  uint8_t* smem = smem_raw;
  if (sb & 1023u) __trap();                       // swizzled TMA / UMMA tiles need 1024 B alignment
  const uint32_t bar0 = sb + SMEM::BAR_OFF;
  const uint32_t q_full = bar0;                                  // [2]
  const uint32_t q_empty = q_full + 2 * 8;                       // [2]
  const uint32_t kb_full = q_empty + 2 * 8;                      // [KB_STAGES]
  const uint32_t kb_empty = kb_full + ATT_KB_STAGES * 8;         // [KB_STAGES]
  const uint32_t v_full = kb_empty + ATT_KB_STAGES * 8;          // [V_STAGES]
  const uint32_t v_empty = v_full + ATT_V_STAGES * 8;            // [V_STAGES]
  const uint32_t s_full = v_empty + ATT_V_STAGES * 8;            // [2]
  const uint32_t p_full = s_full + 2 * 8;                        // [2]
  const uint32_t o_full = p_full + 2 * 8;                        // [1]  every P V commit
  const uint32_t qt_full = o_full + 8;                           // [1]  once per item: Q has been copied into TMEM
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SMEM::BAR_OFF);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + SMEM::N_BARS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // developer trace: role R (0 softmax warp 2 / 1 MMA / 2 producer), tile T, slot K of 8
#define ATT_TRACE(R, T, K)                                                                             \
  if constexpr (kTrace) {                                                                              \
    if (blockIdx.x == 0 && (T) < 96) args.trace[(R) * 1024 + (T) * 8 + (K)] = clock64();              \
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_q);
    tma_prefetch_desc(&tmap_k);
    tma_prefetch_desc(&tmap_vt);
    tma_prefetch_desc(&tmap_bias);
    if constexpr (kSplit) {
      tma_prefetch_desc(&maps.q_lo); tma_prefetch_desc(&maps.k_lo); tma_prefetch_desc(&maps.vt_lo); tma_prefetch_desc(&maps.bias_lo);
    }
    uint64_t* b = bars;
    for (int i = 0; i < 2; ++i) mbar_init(b++, 1);                  // q_full
    for (int i = 0; i < 2; ++i) mbar_init(b++, ATT_SM_WARPS);       // q_empty: the softmax warps copied Q to TMEM
    for (int i = 0; i < 2 * ATT_KB_STAGES; ++i) mbar_init(b++, 1);  // kb_full, kb_empty (S commit)
    for (int i = 0; i < 2 * ATT_V_STAGES; ++i) mbar_init(b++, 1);   // v_full, v_empty (P V commit)
    for (int i = 0; i < 2; ++i) mbar_init(b++, 1);                  // s_full
    for (int i = 0; i < 2; ++i) mbar_init(b++, ATT_SM_WARPS);       // p_full
    mbar_init(b++, 1);                                              // o_full
    mbar_init(b++, ATT_SM_WARPS);                                   // qt_full
    fence_mbar_init();
  }
  // constant rows 64..79 of every V^T tile: row 64 = 1.0 (PV then also yields the row sum of P), rest 0
  for (int i = threadIdx.x; i < ATT_V_STAGES * 128; i += blockDim.x) {
    const int stg = i >> 7, chunk = i & 127;                   // 128 x 16 B chunks = rows 64..79
    uint8_t* base = smem + SMEM::V_OFF + stg * SMEM::V_STAGE + ATT_D * 128;
    const uint32_t val = (chunk < 8) ? 0x3F803F80u : 0u;       // first 8 chunks = row 64
    *reinterpret_cast<uint4*>(base + chunk * 16) = make_uint4(val, val, val, val);
  }
  // fp16 identity [64 keys x 64], K-major SWIZZLE_128B: 16 B chunk c of row n sits at n*128 + ((c ^ (n & 7)) << 4)
  for (int i = threadIdx.x; i < ATT_BKV * 8; i += blockDim.x) {
    const int n = i >> 3, cchunk = i & 7;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    if ((n >> 3) == cchunk) w[(n & 7) >> 1] = (n & 1) ? 0x3C000000u : 0x00003C00u;   // fp16 1.0 at element n
    *reinterpret_cast<uint4*>(smem + SMEM::I_OFF + n * 128 + ((cchunk ^ (n & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
  }
  fence_proxy_async_smem();
  if (warp == 1) tmem_alloc<SMEM::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;            // 2 x 64 columns; P_t (bf16 pairs) overwrites columns [0,32) of S_t
  const uint32_t tmem_O = tmem_base + 128;      // 80 columns: 64 dims + row sum + padding
  const uint32_t tmem_Q = tmem_base + 208;      // 32 columns: the item's Q tile (64 bf16 per row) as the TMEM A operand
  const uint32_t tmem_Qlo = tmem_base + 240;    // kSplit: 32 columns, low part of Q

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (elect_one()) {
      AttCursor c = att_first(total_items, stride, args);
      uint32_t t = 0;
      int loaded_ii = -1;
      int pv_row = 0, pv_kv0 = 0;                 // V^T tile of the previous tile (loaded one tile late, see below)
      constexpr int PF_DIST = 4;                  // L2 prefetch distance in key tiles
      while (c.valid) {
        const int row0 = c.row0;
        if (c.ii != loaded_ii) {
          // Q tiles are loaded ONE ITEM AHEAD: at the first key tile of item ii the producer fetches the Q of item
          // ii + 1 into the other Q buffer (free since the softmax warps copied item ii - 1's Q to TMEM), so that the
          // copy of the next Q to TMEM at the end of this item finds it in shared memory (loaded on arrival at the
          // item, it was ~2500 cycles late: the producer runs only two key tiles ahead of the MMAs)
          loaded_ii = c.ii;
          auto load_q = [&](int k, int qrow, int qhead) {          // Q of this CTA's k-th item -> buffer k & 1
            const int qb = k & 1;
            mbar_wait(q_empty + qb * 8, ((k >> 1) & 1) ^ 1);
            mbar_expect_tx(q_full + qb * 8, SMEM::Q_STAGE);
            tma_load_2d(sb + SMEM::Q_OFF + qb * SMEM::Q_STAGE, &tmap_q, q_full + qb * 8, qhead * ATT_D, qrow);
            if constexpr (kSplit)
              tma_load_2d(sb + SMEM::Q_OFF + qb * SMEM::Q_STAGE + SMEM::Q_BYTES, &maps.q_lo, q_full + qb * 8, qhead * ATT_D, qrow);
          };
          ATT_TRACE(2, t, 2)
          if (c.ii == 0) load_q(0, row0 + c.q0, c.head);
          if (c.nitem < total_items) {
            const int nn_qt = (c.nmeta.y + ATT_BQ - 1) / ATT_BQ;
            const int nlocal = c.nitem - args.heads * c.nmeta.w;
            const int nhead = nlocal / nn_qt;
            load_q(c.ii + 1, c.nmeta.x + (nlocal - nhead * nn_qt) * ATT_BQ, nhead);
          }
        }
        const int kv0 = c.j * ATT_BKV;
        const int brow = (c.doc * args.heads + c.head) * S + c.q0;
        const int vrow = (c.slot * args.heads + c.head) * ATT_D;
        // K + bias of tile t: the stage is free as soon as S_{t-KB_STAGES} has been computed
        const int st = t % ATT_KB_STAGES;
        ATT_TRACE(2, t, 0)
        mbar_wait(kb_empty + st * 8, ((t / ATT_KB_STAGES) & 1) ^ 1);
        ATT_TRACE(2, t, 1)
        const uint32_t sk = sb + SMEM::KB_OFF + st * SMEM::KB_STAGE;
        if (!kSplit && args.experiment && t >= 4) {
          const uint32_t bytes = ((args.experiment & 1) ? 0 : SMEM::K_BYTES) + ((args.experiment & 2) ? 0 : SMEM::B_BYTES);
          if (bytes) mbar_expect_tx(kb_full + st * 8, bytes); else mbar_arrive(kb_full + st * 8);
          if (!(args.experiment & 1)) tma_load_2d(sk, &tmap_k, kb_full + st * 8, args.H + c.head * ATT_D, row0 + kv0);
          if (!(args.experiment & 2)) tma_load_2d(sk + SMEM::NP * SMEM::K_BYTES, &tmap_bias, kb_full + st * 8, kv0, brow);
        } else {
        mbar_expect_tx(kb_full + st * 8, SMEM::KB_STAGE);
        tma_load_2d(sk, &tmap_k, kb_full + st * 8, args.H + c.head * ATT_D, row0 + kv0);
        tma_load_2d(sk + SMEM::NP * SMEM::K_BYTES, &tmap_bias, kb_full + st * 8, kv0, brow);
        }
        if constexpr (kSplit) {
          tma_load_2d(sk + SMEM::K_BYTES, &maps.k_lo, kb_full + st * 8, args.H + c.head * ATT_D, row0 + kv0);
          tma_load_2d(sk + 2 * SMEM::K_BYTES + SMEM::B_BYTES, &maps.bias_lo, kb_full + st * 8, kv0, brow);
        }
        // pull the tiles PF_DIST ahead into L2 (bias always comes from DRAM; K / V^T only for the first query tile
        // of a (slot, head)); one tile per step, so demand loads never queue behind a burst of prefetches
        {
          int pj = c.j + PF_DIST, prow0 = row0, pbrow = brow, pvrow = vrow, phead = c.head, plast = c.last_j;
          if (pj > c.last_j) {                    // runs into the next item of this CTA
            const int nitem = c.nitem;
            if (nitem < total_items) {
              const int nrows = c.nmeta.y;
              const int nn_qt = (nrows + ATT_BQ - 1) / ATT_BQ;
              const int nlocal = nitem - args.heads * c.nmeta.w;
              const int nslot = __ldg(args.qt_slot + nitem / args.heads);
              phead = nlocal / nn_qt;
              pj = pj - c.last_j - 1;
              plast = (nrows + ATT_BKV - 1) / ATT_BKV - 1;
              prow0 = c.nmeta.x;
              pbrow = (c.nmeta.z * args.heads + phead) * S + (nlocal - phead * nn_qt) * ATT_BQ;
              pvrow = (nslot * args.heads + phead) * ATT_D;
            } else {
              pj = plast + 1;
            }
          }
          if (pj <= plast) {
            tma_prefetch_2d(&tmap_bias, pj * ATT_BKV, pbrow);
            tma_prefetch_2d(&tmap_k, args.H + phead * ATT_D, prow0 + pj * ATT_BKV);
            tma_prefetch_2d(&tmap_vt, pj * ATT_BKV, pvrow);
          }
        }
        // V^T of the PREVIOUS tile: it is only needed by P V_{t-1}, which runs a whole softmax later than S_{t-1};
        // loading it after K/bias of tile t keeps the wait for its stage (P V_{t-1-V_STAGES}) off the S path
        if (t > 0) {
          const int sv = (t - 1) % ATT_V_STAGES;
          mbar_wait(v_empty + sv * 8, (((t - 1) / ATT_V_STAGES) & 1) ^ 1);
          if (!kSplit && (args.experiment & 1) && t >= 4) {
            mbar_arrive(v_full + sv * 8);
          } else {
          mbar_expect_tx(v_full + sv * 8, SMEM::NP * ATT_D * ATT_BKV * 2);
          tma_load_2d(sb + SMEM::V_OFF + sv * SMEM::V_STAGE, &tmap_vt, v_full + sv * 8, pv_kv0, pv_row);
          if constexpr (kSplit)
            tma_load_2d(sb + SMEM::V_OFF + sv * SMEM::V_STAGE + SMEM::V_BYTES, &maps.vt_lo, v_full + sv * 8, pv_kv0, pv_row);
          }
        }
        pv_row = vrow; pv_kv0 = kv0;
        ++t;
        c = att_next(c, total_items, stride, args);
      }
      if (t > 0) {
        const int sv = (t - 1) % ATT_V_STAGES;
        mbar_wait(v_empty + sv * 8, (((t - 1) / ATT_V_STAGES) & 1) ^ 1);
        mbar_expect_tx(v_full + sv * 8, SMEM::NP * ATT_D * ATT_BKV * 2);
        tma_load_2d(sb + SMEM::V_OFF + sv * SMEM::V_STAGE, &tmap_vt, v_full + sv * 8, pv_kv0, pv_row);
        if constexpr (kSplit)
          tma_load_2d(sb + SMEM::V_OFF + sv * SMEM::V_STAGE + SMEM::V_BYTES, &maps.vt_lo, v_full + sv * 8, pv_kv0, pv_row);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_bf16(ATT_BQ, ATT_BKV);
      constexpr uint32_t idesc_o = umma_idesc_bf16(ATT_BQ, ATT_DV);
      constexpr uint32_t idesc_s16 = umma_idesc_bf16(ATT_BQ, 16);   // the 16-key tail tile (args.tail_j)
      constexpr uint32_t idesc_b16 = umma_idesc_f16(ATT_BQ, 16);
      const uint64_t di = umma_desc_sw128_kmajor(sb + SMEM::I_OFF);
      AttCursor cs = att_first(total_items, stride, args);   // next S = Q K^T + B I to issue (one tile ahead)
      AttCursor cp = cs;                                              // next P V to issue
      uint32_t ts = 0;
      auto issue_s = [&]() {
        const int st = ts % ATT_KB_STAGES;
        ATT_TRACE(1, ts, 0)
        if (cs.j == 0) mbar_wait(qt_full, cs.ii & 1);               // the item's Q is in TMEM (softmax warps, below)
        mbar_wait(kb_full + st * 8, (ts / ATT_KB_STAGES) & 1);
        ATT_TRACE(1, ts, 1)
        tc_fence_after();
        const uint32_t stage = sb + SMEM::KB_OFF + st * SMEM::KB_STAGE;
        const uint64_t dk = umma_desc_sw128_kmajor(stage);
        const uint64_t db = umma_desc_sw128_kmajor(stage + SMEM::NP * SMEM::K_BYTES);
        const uint32_t d_s = tmem_S + (ts & 1) * ATT_BKV;
        // S buffer ts&1 last held P_{ts-2}; its P V was issued before this point and tcgen05.mma executes in order
        if constexpr (kSplit) {
          // S = Q_hi K_hi^T + Q_lo K_hi^T + Q_hi K_lo^T + B_hi I + B_lo I   (the 16-key tail path is off in this mode)
          const uint64_t dkl = umma_desc_sw128_kmajor(stage + SMEM::K_BYTES);
          const uint64_t dbl = umma_desc_sw128_kmajor(stage + 2 * SMEM::K_BYTES + SMEM::B_BYTES);
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k) umma_bf16_ts(d_s, tmem_Q + k * 8, dk + 2 * k, idesc_s, k ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k) umma_bf16_ts(d_s, tmem_Qlo + k * 8, dk + 2 * k, idesc_s, 1u);
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k) umma_bf16_ts(d_s, tmem_Q + k * 8, dkl + 2 * k, idesc_s, 1u);
          // bias x identity, block-diagonal (see the bf16 path below)
#pragma unroll
          for (int k = 0; k < ATT_BKV / 16; ++k) umma_bf16_ss(d_s + 16 * k, db + 2 * k, di + 130 * k, idesc_b16, 1u);
#pragma unroll
          for (int k = 0; k < ATT_BKV / 16; ++k) umma_bf16_ss(d_s + 16 * k, dbl + 2 * k, di + 130 * k, idesc_b16, 1u);
        } else if (cs.j != cs.tail_j) {
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k) umma_bf16_ts(d_s, tmem_Q + k * 8, dk + 2 * k, idesc_s, k ? 1u : 0u);
          // += bias16 x I, block by block: key block k of the bias tile only meets the k-th 16 x 16 diagonal block of
          // the identity, so each of the four MMAs has N = 16 (output columns 16k .. 16k + 15) instead of N = 64: a
          // quarter of the tensor-pipe time, the same bits (the off-diagonal blocks only ever added exact zeros), and
          // the four no longer form a dependent chain on one accumulator.  Identity rows 16k .. at byte 2048 k (two
          // 8-row swizzle atoms), its K block k at +32 k bytes: descriptor + 128 k + 2 k.
#pragma unroll
          for (int k = 0; k < ATT_BKV / 16; ++k) umma_bf16_ss(d_s + 16 * k, db + 2 * k, di + 130 * k, idesc_b16, 1u);
        } else {
          // only keys 0..15 of the tile exist: N = 16 (K rows 0..15, bias columns 0..15, one identity block)
#pragma unroll
          for (int k = 0; k < ATT_D / 16; ++k) umma_bf16_ts(d_s, tmem_Q + k * 8, dk + 2 * k, idesc_s16, k ? 1u : 0u);
          umma_bf16_ss(d_s, db, di, idesc_b16, 1u);
        }
        umma_commit(s_full + (ts & 1) * 8);
        umma_commit(kb_empty + st * 8);
        ++ts;
        cs = att_next(cs, total_items, stride, args);
      };
      if (cs.valid) issue_s();
      for (uint32_t t = 0; t < ts; ++t) {               // ts grows while tiles remain
        if (cs.valid) issue_s();                        // S_{t+1} (its TMEM buffer was released by P V_{t-1} above)
        const int sv = t % ATT_V_STAGES;
        const int b = t & 1;
        const bool first = (cp.j == 0);
        // P_t is in TMEM; for the first tile of an item the softmax warps have also read the previous item's O
        ATT_TRACE(1, t, 2)
        mbar_wait(p_full + b * 8, (t >> 1) & 1);
        ATT_TRACE(1, t, 3)
        mbar_wait(v_full + sv * 8, (t / ATT_V_STAGES) & 1);
        tc_fence_after();
        const uint64_t dv = umma_desc_sw128_kmajor(sb + SMEM::V_OFF + sv * SMEM::V_STAGE);
        const int pv_steps = (kSplit || cp.j != cp.tail_j) ? ATT_BKV / 16 : 1;        // tail tile: P is [128 x 16]
#pragma unroll
        for (int k = 0; k < ATT_BKV / 16; ++k)
          if (k < pv_steps)
            umma_bf16_ts(tmem_O, tmem_S + b * ATT_BKV + k * 8, dv + 2 * k, idesc_o, (k || !first) ? 1u : 0u);
        if constexpr (kSplit) {
          // O += P_lo [V_hi | 1] + P_hi V_lo   (P_lo sits in columns [32, 64) of the S buffer; V_lo has no ones row)
          constexpr uint32_t idesc_o64 = umma_idesc_bf16(ATT_BQ, ATT_D);
          const uint64_t dvl = umma_desc_sw128_kmajor(sb + SMEM::V_OFF + sv * SMEM::V_STAGE + SMEM::V_BYTES);
#pragma unroll
          for (int k = 0; k < ATT_BKV / 16; ++k) umma_bf16_ts(tmem_O, tmem_S + b * ATT_BKV + 32 + k * 8, dv + 2 * k, idesc_o, 1u);
#pragma unroll
          for (int k = 0; k < ATT_BKV / 16; ++k) umma_bf16_ts(tmem_O, tmem_S + b * ATT_BKV + k * 8, dvl + 2 * k, idesc_o64, 1u);
        }
        umma_commit(o_full);
        umma_commit(v_empty + sv * 8);
        cp = att_next(cp, total_items, stride, args);
      }
    }
  } else {
    // ------------------------------------------------------------ softmax (warps 2..5), thread = query row
    const int quarter = warp & 3;                             // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;                        // query row within the tile == TMEM lane
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    uint32_t t = 0;
    AttCursor c = att_first(total_items, stride, args);

    float ref = 0.f, alpha_pend = 1.f;
    __nv_bfloat16* out_ptr = nullptr;                         // ctx destination of the open item (nullptr: row >= S)
    bool have_item = false;

    // O (TMEM) / row sum -> ctx[row, head*64 .. +63]; the caller has waited for the item's last P V
    auto store_item = [&](__nv_bfloat16* dst_row) {
      uint32_t v[32];
      const uint32_t lsum = tmem_ld1(tmem_O + lane_addr + ATT_D);
      tmem_ld32(tmem_O + lane_addr, v);
      tmem_ld_wait();
      const float inv = 1.0f / __uint_as_float(lsum);
      if constexpr (kSplit) {
        // ctx as a split pair: hi = bf16(o / l), lo = bf16(o / l - hi)
        __nv_bfloat16* lo_row = dst_row ? args.ctx_lo + (dst_row - args.ctx) : nullptr;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          if (hh) { tmem_ld32(tmem_O + lane_addr + 32, v); tmem_ld_wait(); }
          if (dst_row) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              uint32_t h[4], l[4];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float a = __uint_as_float(v[i * 8 + 2 * j]) * inv, c2 = __uint_as_float(v[i * 8 + 2 * j + 1]) * inv;
                h[j] = pack_bf16x2(a, c2);
                const float2 hf = unpack_bf16x2(h[j]);
                l[j] = pack_bf16x2(a - hf.x, c2 - hf.y);
              }
              reinterpret_cast<uint4*>(dst_row)[hh * 4 + i] = make_uint4(h[0], h[1], h[2], h[3]);
              reinterpret_cast<uint4*>(lo_row)[hh * 4 + i] = make_uint4(l[0], l[1], l[2], l[3]);
            }
          }
        }
        return;
      }
      uint4* dst = reinterpret_cast<uint4*>(dst_row);
      if (dst_row) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dst[i] = make_uint4(pack_bf16x2(__uint_as_float(v[i * 8 + 0]) * inv, __uint_as_float(v[i * 8 + 1]) * inv),
                              pack_bf16x2(__uint_as_float(v[i * 8 + 2]) * inv, __uint_as_float(v[i * 8 + 3]) * inv),
                              pack_bf16x2(__uint_as_float(v[i * 8 + 4]) * inv, __uint_as_float(v[i * 8 + 5]) * inv),
                              pack_bf16x2(__uint_as_float(v[i * 8 + 6]) * inv, __uint_as_float(v[i * 8 + 7]) * inv));
      }
      tmem_ld32(tmem_O + lane_addr + 32, v);
      tmem_ld_wait();
      if (dst_row) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          dst[4 + i] = make_uint4(pack_bf16x2(__uint_as_float(v[i * 8 + 0]) * inv, __uint_as_float(v[i * 8 + 1]) * inv),
                                  pack_bf16x2(__uint_as_float(v[i * 8 + 2]) * inv, __uint_as_float(v[i * 8 + 3]) * inv),
                                  pack_bf16x2(__uint_as_float(v[i * 8 + 4]) * inv, __uint_as_float(v[i * 8 + 5]) * inv),
                                  pack_bf16x2(__uint_as_float(v[i * 8 + 6]) * inv, __uint_as_float(v[i * 8 + 7]) * inv));
      }
    };

    // Q of item `ii` : smem (TMA, SW128) -> this thread's row -> TMEM A operand.  Read once per item instead of by
    // every Q.K^T MMA (16 KB of shared-memory reads per key tile less).  Called when no S MMA of the previous item is
    // pending any more (its last s_full has been waited on).
    auto q_to_tmem = [&](int ii) {
      const int qb = ii & 1;
      mbar_wait(q_full + qb * 8, (ii >> 1) & 1);
      const uint32_t qrow = sb + SMEM::Q_OFF + qb * SMEM::Q_STAGE + r * 128;
      uint32_t q[32];
#pragma unroll
      for (int cch = 0; cch < 8; ++cch) {
        const uint4 x = lds128(qrow + ((cch ^ (r & 7)) << 4));
        q[4 * cch] = x.x; q[4 * cch + 1] = x.y; q[4 * cch + 2] = x.z; q[4 * cch + 3] = x.w;
      }
      tmem_st32(tmem_Q + lane_addr, q);
      if constexpr (kSplit) {
#pragma unroll
        for (int cch = 0; cch < 8; ++cch) {
          const uint4 x = lds128(qrow + SMEM::Q_BYTES + ((cch ^ (r & 7)) << 4));
          q[4 * cch] = x.x; q[4 * cch + 1] = x.y; q[4 * cch + 2] = x.z; q[4 * cch + 3] = x.w;
        }
        tmem_st32(tmem_Qlo + lane_addr, q);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(qt_full); mbar_arrive(q_empty + qb * 8); }
    };
    if (c.valid) q_to_tmem(0);

    while (c.valid) {
      const int b = t & 1;
      const bool first = (c.j == 0);                         // first key tile of a new item
      const uint32_t tS = tmem_S + lane_addr + b * ATT_BKV;
      __nv_bfloat16* prev_out = out_ptr;
      if (first) {
        const int q = c.q0 + r;
        out_ptr = (q < c.rows) ? args.ctx + static_cast<size_t>(c.row0 + q) * args.H + c.head * ATT_D : nullptr;
      }
      const bool tr = kTrace && warp == 2 && lane == 0;
      if (tr) { ATT_TRACE(0, t, 0) }
      mbar_wait(s_full + b * 8, (t >> 1) & 1);      // S_t = Q K^T + bias (+ key mask) is complete
      tc_fence_after();
      if (tr) { ATT_TRACE(0, t, 1) }
      // last tile of this item: every S MMA that reads the item's Q has completed -> stage the next item's Q
      if (c.j == c.last_j && c.nitem < total_items) q_to_tmem(c.ii + 1);

      float pmax;
      if constexpr (kSplit) {
        // fp32 mode: P as a split pair, P_hi (bf16 pairs) in columns [0, 32) and P_lo = bf16(p - P_hi) in [32, 64) of
        // the S buffer (the row's 64 scores are in registers by then).  Reference handling as in the bf16 path below.
        uint32_t v0[32], v1[32], ph[32], pl[32];
        tmem_ld32(tS, v0);
        tmem_ld32(tS + 32, v1);
        tmem_ld_wait();
        if (first) {
          float m0 = fmaxf(__uint_as_float(v0[0]), __uint_as_float(v0[1]));
#pragma unroll
          for (int i = 2; i < 32; i += 2) m0 = fmaxf(m0, fmaxf(__uint_as_float(v0[i]), __uint_as_float(v0[i + 1])));
#pragma unroll
          for (int i = 0; i < 32; i += 2) m0 = fmaxf(m0, fmaxf(__uint_as_float(v1[i]), __uint_as_float(v1[i + 1])));
          ref = m0;
        }
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const float a0 = __uint_as_float(i < 16 ? v0[2 * i] : v1[2 * i - 32]) - ref;
          const float a1 = __uint_as_float(i < 16 ? v0[2 * i + 1] : v1[2 * i - 31]) - ref;
          m = fmaxf(m, fmaxf(a0, a1));
          const float e0 = fast_exp2(a0), e1 = fast_exp2(a1);
          ph[i] = pack_bf16x2(e0, e1);
          const float2 hf = unpack_bf16x2(ph[i]);
          pl[i] = pack_bf16x2(e0 - hf.x, e1 - hf.y);
        }
        pmax = m;
        if (pmax > ATT_JUMP) {
          const float dq = ceilf(pmax);
          ref += dq;
          alpha_pend *= fast_exp2(-dq);
          pmax -= dq;
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float e0 = fast_exp2(__uint_as_float(i < 16 ? v0[2 * i] : v1[2 * i - 32]) - ref);
            const float e1 = fast_exp2(__uint_as_float(i < 16 ? v0[2 * i + 1] : v1[2 * i - 31]) - ref);
            ph[i] = pack_bf16x2(e0, e1);
            const float2 hf = unpack_bf16x2(ph[i]);
            pl[i] = pack_bf16x2(e0 - hf.x, e1 - hf.y);
          }
        }
        __syncwarp();
        tmem_st32(tS, ph);
        tmem_st32(tS + 32, pl);
      } else if (c.j == c.tail_j) {
        // 16-key tail tile: a quarter of the loads, exponentials and stores
        uint32_t v[16], pq[8];
        tmem_ld16(tS, v);
        tmem_ld_wait();
        if (tr) { ATT_TRACE(0, t, 2) }
        if (first) {
          float m = fmaxf(__uint_as_float(v[0]), __uint_as_float(v[1]));
#pragma unroll
          for (int i = 2; i < 16; i += 2) m = fmaxf(m, fmaxf(__uint_as_float(v[i]), __uint_as_float(v[i + 1])));
          ref = m;
        }
        float m = -INFINITY;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float a0 = __uint_as_float(v[2 * i]) - ref, a1 = __uint_as_float(v[2 * i + 1]) - ref;
          m = fmaxf(m, fmaxf(a0, a1));
          pq[i] = pack_bf16x2(fast_exp2(a0), fast_exp2(a1));
        }
        pmax = m;
        if (pmax > ATT_JUMP) {                       // see the full-tile path below
          const float dq = ceilf(pmax);
          ref += dq;
          alpha_pend *= fast_exp2(-dq);
          pmax -= dq;
#pragma unroll
          for (int i = 0; i < 8; ++i)
            pq[i] = pack_bf16x2(fast_exp2(__uint_as_float(v[2 * i]) - ref), fast_exp2(__uint_as_float(v[2 * i + 1]) - ref));
        }
        __syncwarp();
        tmem_st8(tS, pq);
      } else {
        uint32_t v0[32], v1[32], pk[32];
        tmem_ld32(tS, v0);
        tmem_ld32(tS + 32, v1);
        tmem_ld_wait();
        if (tr) { ATT_TRACE(0, t, 2) }
        if (first) {
          // exact row maximum of the first tile as the reference, then p = exp2(s - ref)
          float m0 = fmaxf(__uint_as_float(v0[0]), __uint_as_float(v0[1]));
          float m1 = fmaxf(__uint_as_float(v1[0]), __uint_as_float(v1[1]));
#pragma unroll
          for (int i = 2; i < 32; i += 2) {
            m0 = fmaxf(m0, fmaxf(__uint_as_float(v0[i]), __uint_as_float(v0[i + 1])));
            m1 = fmaxf(m1, fmaxf(__uint_as_float(v1[i]), __uint_as_float(v1[i + 1])));
          }
          ref = fmaxf(m0, m1);
          pmax = 0.f;
        }
        {
          // p = exp2(s - ref); the running max rides along (FMNMX on the ALU pipe, MUFU on the XU pipe)
          float m0 = -INFINITY, m1 = -INFINITY;
          uint64_t nref2;
          asm("mov.b64 %0, {%1, %1};" : "=l"(nref2) : "f"(-ref));
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float a0, a1, c0, c1;                       // s - ref, two per packed-fp32 instruction (FADD2)
            sub_ref_x2(v0[2 * i], v0[2 * i + 1], nref2, a0, a1);
            sub_ref_x2(v1[2 * i], v1[2 * i + 1], nref2, c0, c1);
            m0 = fmaxf(m0, fmaxf(a0, a1));
            m1 = fmaxf(m1, fmaxf(c0, c1));
            pk[i] = pack_bf16x2(fast_exp2(a0), fast_exp2(a1));
            pk[16 + i] = pack_bf16x2(fast_exp2(c0), fast_exp2(c1));
          }
          pmax = fmaxf(m0, m1);
        }
        if (pmax > ATT_JUMP) {
          // a score of this tile is more than 2^40 above the row reference (never at init, possible with sharp trained
          // heads): raise the reference NOW, recompute this row's P against it and fold the factor into the rescale of
          // O below, so no probability ever leaves the fp32 / bf16 range
          const float dq = ceilf(pmax);
          ref += dq;
          alpha_pend *= fast_exp2(-dq);
          pmax -= dq;
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            pk[i] = pack_bf16x2(fast_exp2(__uint_as_float(v0[2 * i]) - ref), fast_exp2(__uint_as_float(v0[2 * i + 1]) - ref));
            pk[16 + i] = pack_bf16x2(fast_exp2(__uint_as_float(v1[2 * i]) - ref), fast_exp2(__uint_as_float(v1[2 * i + 1]) - ref));
          }
        }
        __syncwarp();
        tmem_st32(tS, pk);
      }
      if (tr) { ATT_TRACE(0, t, 3) }

      // ---- P V_{t-1} must be complete before O is read (new item) or rescaled, and before P V_t may be issued
      if (t > 0) {
        mbar_wait(o_full, (t - 1) & 1);
        tc_fence_after();
        if (tr) { ATT_TRACE(0, t, 4) }
        if (first) {
          if (have_item) store_item(prev_out);
        } else if (__any_sync(0xffffffffu, alpha_pend != 1.0f)) {    // rare: an earlier tile raised the row reference
          uint32_t o[32];
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) {
            tmem_ld32(tmem_O + lane_addr + hh * 32, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha_pend);
            tmem_st32(tmem_O + lane_addr + hh * 32, o);
          }
          const uint32_t ls = tmem_ld1(tmem_O + lane_addr + ATT_D);
          tmem_ld_wait();
          tmem_st1(tmem_O + lane_addr + ATT_D, __float_as_uint(__uint_as_float(ls) * alpha_pend));
        }
      }
      have_item = true;
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full + b * 8);
      if (tr) { ATT_TRACE(0, t, 5) }

      // ---- reference for the following tiles (lazy: only when a score ran more than 2^8 above it)
      alpha_pend = 1.f;
      if (pmax > ATT_LAZY) {
        const float dq = ceilf(pmax);
        ref += dq;
        alpha_pend = fast_exp2(-dq);
        if (!(alpha_pend > 0.f)) *args.err_flag = 1;       // unreachable with the jump handling above; kept as a guard
      }
      ++t;
      c = att_next(c, total_items, stride, args);
    }
    if (have_item) {
      mbar_wait(o_full, (t - 1) & 1);
      tc_fence_after();
      store_item(out_ptr);
    }
  }

#undef ATT_TRACE
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<SMEM::TMEM_COLS>(tmem_base);
  }
}

// ------------------------------------------------------------------ host side: tensor maps, launch
// The engine and the attention tests (tests/kernels/attention_harness.cu) both launch through these, so the tests run
// the engine's own launch.

// The maps of the layouts above over m_rows rows of qk and `docs` documents (V^T by slot, the bias by document).
// split (fp32 engine mode): the *_lo pointers are the low parts; otherwise they are ignored and lo = hi.
inline AttMaps attention_maps(const void* qk, const void* qk_lo, const void* vt, const void* vt_lo, const void* bias,
                              const void* bias_lo, uint64_t m_rows, int H, int heads, int seq, int docs, int kv_pitch,
                              int bias_pitch, bool split) {
  const uint64_t vt_rows = static_cast<uint64_t>(docs) * heads * 64, bias_rows = static_cast<uint64_t>(docs) * heads * seq;
  auto make = [&](const void* q, const void* v, const void* b, CUtensorMap& mq, CUtensorMap& mk, CUtensorMap& mv,
                  CUtensorMap& mb) {
    mq = make_tmap_2d_sw128(q, m_rows, 2 * H, 2 * H, ATT_BQ);
    mk = make_tmap_2d_sw128(q, m_rows, 2 * H, 2 * H, ATT_BKV);
    mv = make_tmap_2d_sw128(v, vt_rows, kv_pitch, kv_pitch, 64);
    mb = make_tmap_2d_sw128(b, bias_rows, bias_pitch, bias_pitch, ATT_BQ, CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  };
  AttMaps m;
  make(qk, vt, bias, m.q, m.k, m.vt, m.bias);
  if (split) make(qk_lo, vt_lo, bias_lo, m.q_lo, m.k_lo, m.vt_lo, m.bias_lo);
  else { m.q_lo = m.q; m.k_lo = m.k; m.vt_lo = m.vt; m.bias_lo = m.bias; }
  return m;
}

// One attention launch on `device` (an ordinal, passed in so a launch queries nothing) with `sms` SMs: ATT_CTAS_PER_SM
// CTAs per SM, or one for split (the fp32-mode kernel) and for one_cta (bf16: 16 KB of extra dynamic shared memory
// keep a second CTA off the SM).  trace (bf16): the kTrace instantiation.  Static (internal linkage): every library
// built from this header (the engine, a test harness) keeps its own attribute cache for its own copy of the kernels.
static inline void launch_attention(int device, int sms, const AttMaps& maps, const AttArgs& args, bool split, bool trace,
                                    bool one_cta, cudaStream_t st) {
  // the shared-memory attribute is per device; it is set by the first launch, before a plan captures a forward
  static bool configured[64] = {};
  if (!configured[device & 63]) {
    CUDA_OK(cudaFuncSetAttribute(attention_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmem::DYN_BYTES + 16 * 1024));
    CUDA_OK(cudaFuncSetAttribute(attention_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmem::DYN_BYTES + 16 * 1024));
    CUDA_OK(cudaFuncSetAttribute(attention_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmemT<true>::DYN_BYTES));
    configured[device & 63] = true;
  }
  const int grid = sms * ((split || one_cta) ? 1 : ATT_CTAS_PER_SM);
  const size_t smem = AttSmem::DYN_BYTES + (one_cta ? 16 * 1024 : 0);
  if (split)
    attention_kernel<false, true><<<grid, ATT_THREADS, AttSmemT<true>::DYN_BYTES, st>>>(maps, args);
  else if (trace)
    attention_kernel<true, false><<<grid, ATT_THREADS, smem, st>>>(maps, args);
  else
    attention_kernel<false, false><<<grid, ATT_THREADS, smem, st>>>(maps, args);
  CUDA_OK(cudaGetLastError());
}

}  // namespace mmee
