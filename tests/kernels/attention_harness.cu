// Stand-alone launcher of the fused attention kernel (csrc/attention.cuh) and of the row planner (plan_rows_kernel,
// csrc/norm_exit.cuh) on caller-built inputs, for tests/test_attention_gpu.py.  Test-only code: the engine never links
// it.  All pointers are device pointers (torch tensors); both calls synchronise and return a cudaError_t (0 = success).
//
// The tensor maps, the shared-memory attribute, the grid and the launch are literal copies of the engine's lines
// (engine.cu, allocate(): t_qk / t_k64 / t_vt / t_bias; forward_device(): the attention launch of an encoder layer),
// so the kernel sees exactly the operands it sees inside a forward.  When the attention kernel or its launch changes,
// this file changes with it.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <stdexcept>
#include <string>

#include "attention.cuh"
#include "norm_exit.cuh"
#include "tmap.h"

using namespace mmee;

#define CUDA_OK(x)                                                                                   \
  do {                                                                                               \
    cudaError_t e_ = (x);                                                                            \
    if (e_ != cudaSuccess)                                                                           \
      throw std::runtime_error(std::string(#x) + ": " + cudaGetErrorString(e_) + " @" + std::to_string(__LINE__)); \
  } while (0)

extern "C" {

// engine.cu forward_device(): plan_rows_kernel<<<1, 256, 0, st>>>(slot_doc, doc_len, n_dev + stage, plan_view(e, rp),
// m_dev + stage, ATT_BQ).  n_dev: device int, the number of slots.
int att_plan(const int* slot_doc, const int* doc_len, const int* n_dev, int* row0, int* meta, int* qt_slot, int* n_qt,
             int* m_dev) {
  SlotRows r;
  r.row0 = row0;
  r.meta = reinterpret_cast<int4*>(meta);
  r.qt_slot = qt_slot;
  r.n_qt_dev = n_qt;
  plan_rows_kernel<<<1, 256>>>(slot_doc, doc_len, n_dev, r, m_dev, ATT_BQ);
  cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess) err = cudaDeviceSynchronize();
  return static_cast<int>(err);
}

// One attention launch over the work list written by att_plan.
//   qk   bf16 [m_rows, 2H]                      Q (log2 domain) in columns [h*64, h*64+64), K at H + h*64
//   vt   bf16 [n_docs * heads * 64, kv_pitch]   V^T by SLOT, columns = kept-token rank
//   bias fp16 [n_docs * heads * seq, bias_pitch] by DOCUMENT (the mask rides in it as -60000)
//   ctx  bf16 [m_rows, H]
// split != 0: the fp32-mode kernel (attention_kernel<false, true>) with the *_lo low parts; otherwise they are ignored.
// one_cta != 0 (bf16 kernel only): one CTA per SM with 16 KB of extra dynamic shared memory (MMEE_ATT_ONE_CTA).
int att_run(const void* qk, const void* qk_lo, const void* vt, const void* vt_lo, const void* bias, const void* bias_lo,
            void* ctx, void* ctx_lo, const int* meta, const int* qt_slot, const int* n_qt, int* err_flag, int m_rows,
            int H, int heads, int seq, int n_docs, int kv_pitch, int bias_pitch, int tail16, int split, int one_cta) {
  try {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int B = n_docs, S = seq, bias_width = bias_pitch;
    const uint64_t M = static_cast<uint64_t>(m_rows);
    // engine.cu allocate()
    const CUtensorMap t_qk = make_tmap_2d_sw128(qk, M, 2 * H, 2 * H, 128);
    const CUtensorMap t_vt = make_tmap_2d_sw128(vt, static_cast<uint64_t>(B) * heads * 64, kv_pitch, kv_pitch, 64);
    const CUtensorMap t_k64 = make_tmap_2d_sw128(qk, M, 2 * H, 2 * H, ATT_BKV);
    const CUtensorMap t_bias = make_tmap_2d_sw128(bias, static_cast<uint64_t>(B) * heads * S, bias_width, bias_pitch, ATT_BQ,
                                                  CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    CUtensorMap t_qk_lo = t_qk, t_k64_lo = t_k64, t_vt_lo = t_vt, t_bias_lo = t_bias;
    if (split) {
      t_qk_lo = make_tmap_2d_sw128(qk_lo, M, 2 * H, 2 * H, 128);
      t_k64_lo = make_tmap_2d_sw128(qk_lo, M, 2 * H, 2 * H, ATT_BKV);
      t_vt_lo = make_tmap_2d_sw128(vt_lo, static_cast<uint64_t>(B) * heads * 64, kv_pitch, kv_pitch, 64);
      t_bias_lo = make_tmap_2d_sw128(bias_lo, static_cast<uint64_t>(B) * heads * S, bias_width, bias_pitch, ATT_BQ,
                                     CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
    }
    // engine.cu forward_device(), attention of an encoder layer
    AttArgs aa{};
    aa.slot_meta = reinterpret_cast<const int4*>(meta); aa.qt_slot = qt_slot; aa.n_qt_dev = n_qt;
    aa.ctx = static_cast<__nv_bfloat16*>(ctx); aa.ctx_lo = static_cast<__nv_bfloat16*>(ctx_lo); aa.H = H; aa.heads = heads; aa.seq = S;
    aa.tail16 = (tail16 && !split) ? 1 : 0;
    aa.experiment = 0; aa.err_flag = err_flag; aa.trace = nullptr;
    CUDA_OK(cudaFuncSetAttribute(attention_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmem::DYN_BYTES + 16 * 1024));
    CUDA_OK(cudaFuncSetAttribute(attention_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, AttSmemT<true>::DYN_BYTES));
    AttMaps am;
    am.q = t_qk; am.k = t_k64; am.vt = t_vt; am.bias = t_bias;
    if (split) { am.q_lo = t_qk_lo; am.k_lo = t_k64_lo; am.vt_lo = t_vt_lo; am.bias_lo = t_bias_lo; }
    else { am.q_lo = t_qk; am.k_lo = t_k64; am.vt_lo = t_vt; am.bias_lo = t_bias; }
    const int att_grid = sms * ((split || one_cta) ? 1 : ATT_CTAS_PER_SM);
    const size_t att_smem = AttSmem::DYN_BYTES + (one_cta ? 16 * 1024 : 0);
    if (split)
      attention_kernel<false, true><<<att_grid, ATT_THREADS, AttSmemT<true>::DYN_BYTES>>>(am, aa);
    else
      attention_kernel<false, false><<<att_grid, ATT_THREADS, att_smem>>>(am, aa);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaDeviceSynchronize());
    return 0;
  } catch (const std::exception& ex) {
    fprintf(stderr, "att_run: %s\n", ex.what());
    return -1;
  }
}

}  // extern "C"
