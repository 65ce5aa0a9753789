// Stand-alone launcher of the fused attention kernel (csrc/attention.cuh) and of the row planner (plan_rows_kernel,
// csrc/norm_exit.cuh) on caller-built inputs, for tests/test_attention_gpu.py.  Test-only code: the engine never links
// it.  All pointers are device pointers (torch tensors); both calls synchronise and return a cudaError_t (0 = success).
//
// Argument marshalling only: the tensor maps (attention_maps) and the launches (launch_attention, launch_plan_rows)
// are the engine's own, from the host-side sections of attention.cuh and norm_exit.cuh.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <stdexcept>
#include <string>

#include "attention.cuh"
#include "norm_exit.cuh"
#include "tmap.h"

using namespace mmee;

extern "C" {

// The row plan of the encoder's first stage.  n_dev: device int, the number of slots.
int att_plan(const int* slot_doc, const int* doc_len, const int* n_dev, int* row0, int* meta, int* qt_slot, int* n_qt,
             int* m_dev) {
  SlotRows r;
  r.row0 = row0;
  r.meta = reinterpret_cast<int4*>(meta);
  r.qt_slot = qt_slot;
  r.n_qt_dev = n_qt;
  launch_plan_rows(slot_doc, doc_len, n_dev, r, m_dev, ATT_BQ, 0);
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
    CUDA_OK(cudaGetDevice(&dev));
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const AttMaps am = attention_maps(qk, qk_lo, vt, vt_lo, bias, bias_lo, static_cast<uint64_t>(m_rows), H, heads, seq,
                                      n_docs, kv_pitch, bias_pitch, split);
    AttArgs aa{};
    aa.slot_meta = reinterpret_cast<const int4*>(meta); aa.qt_slot = qt_slot; aa.n_qt_dev = n_qt;
    aa.ctx = static_cast<__nv_bfloat16*>(ctx); aa.ctx_lo = static_cast<__nv_bfloat16*>(ctx_lo); aa.H = H; aa.heads = heads; aa.seq = seq;
    aa.tail16 = (tail16 && !split) ? 1 : 0;
    aa.experiment = 0; aa.err_flag = err_flag; aa.trace = nullptr;
    launch_attention(dev, sms, am, aa, split, false, one_cta, 0);
    CUDA_OK(cudaDeviceSynchronize());
    return 0;
  } catch (const std::exception& ex) {
    fprintf(stderr, "att_run: %s\n", ex.what());
    return -1;
  }
}

}  // extern "C"
