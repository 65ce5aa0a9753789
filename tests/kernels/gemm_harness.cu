// Stand-alone launcher of the tcgen05 GEMM (csrc/gemm.cuh) on caller-built inputs, for tests/test_gemm_gpu.py.
// Test-only code: the engine never links it.  All pointers are device pointers (torch tensors); the call synchronises
// and returns a cudaError_t (0 = success; -1 = a host-side failure, printed to stderr).
//
// Argument marshalling only: the tensor maps (gemm_a_map, gemm_w_map), the shape rules and the launch (launch_gemm)
// are the engine's own, from the host-side section of gemm.cuh.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <stdexcept>
#include <string>

#include "gemm.cuh"
#include "tmap.h"

using namespace mmee;

extern "C" {

// The engine's shape rules (gemm.cuh): BLOCK_N of a GEMM family, of the QKV GEMM, and the fp32-mode MLP-down K chunk.
int gemm_bn(int n) { return gemm_block_n(n); }
int gemm_bn_qkv(int H) { return gemm_block_n_qkv(H); }
int gemm_k_chunk(int I) { return gemm_kchunk(I); }

// One GEMM launch: C[M, N] = A[M, K] W[N, K]^T + the epilogue `epi` (GemmEpilogue).
//   a, a_lo  bf16, a_rows rows of K columns at row pitch a_pitch (the A tensor map; the K-chunk maps pass a pointer
//            to column c * kchunk and a_pitch = I).  a_rows is the map's row count, independent of M.
//   w, w_lo  bf16 [N, K] at row pitch w_pitch.
//   bn       128: gemm_tc_kernel<128>, 256: gemm_tc_pair_kernel.  split != 0: fp32 mode (a_lo, w_lo used).
//   grid     0: the engine's grid.
// The remaining arguments are the GemmArgs fields, in the struct's order.
int gemm_run(int epi, int bn, int split, int grid, const void* a, const void* a_lo, long long a_rows, long long a_pitch,
             const void* w, const void* w_lo, long long w_pitch,
             const int* m_dev, int m_static, int N, int K, const float* bias, void* out, void* out_lo, int ld_out,
             const void* resid, const void* resid_lo, const float* resid_f32, const float* resid_y,
             const void* resid_stats, const int* resid_src, const float* resid_w, const float* resid_b,
             int resid_prefetch, void* vt, void* vt_lo, int qk_cols, const int* row0, const int* n_slots_dev,
             int kv_pitch, int heads, const float* pos, int n_patch, int n_vis) {
  try {
    int dev = 0, sms = 0;
    CUDA_OK(cudaGetDevice(&dev));
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    using bf16 = __nv_bfloat16;
    const CUtensorMap ta = gemm_a_map(static_cast<const bf16*>(a), a_rows, K, a_pitch);
    const CUtensorMap tb = gemm_w_map(static_cast<const bf16*>(w), N, K, w_pitch, bn);
    CUtensorMap ta_lo = ta, tb_lo = tb;
    if (split) {
      ta_lo = gemm_a_map(static_cast<const bf16*>(a_lo), a_rows, K, a_pitch);
      tb_lo = gemm_w_map(static_cast<const bf16*>(w_lo), N, K, w_pitch, bn);
    }
    GemmArgs ga{};
    ga.m_dev = m_dev; ga.m_static = m_static; ga.N = N; ga.K = K; ga.bias = bias;
    ga.out = out; ga.out_lo = static_cast<bf16*>(out_lo); ga.ld_out = ld_out;
    ga.resid = static_cast<const bf16*>(resid); ga.resid_lo = static_cast<const bf16*>(resid_lo);
    ga.resid_f32 = resid_f32;
    ga.resid_y = resid_y; ga.resid_stats = static_cast<const float2*>(resid_stats); ga.resid_src = resid_src;
    ga.resid_w = resid_w; ga.resid_b = resid_b; ga.resid_prefetch = resid_prefetch;
    ga.vt = static_cast<bf16*>(vt); ga.vt_lo = static_cast<bf16*>(vt_lo); ga.qk_cols = qk_cols;
    ga.row0 = row0; ga.n_slots_dev = n_slots_dev; ga.kv_pitch = kv_pitch; ga.heads = heads;
    ga.pos = pos; ga.n_patch = n_patch; ga.n_vis = n_vis;
    switch (epi) {
      case EPI_BIAS_BF16: launch_gemm<EPI_BIAS_BF16>(dev, sms, bn, split, ta, tb, ta_lo, tb_lo, ga, 0, grid); break;
      case EPI_GELU_BF16: launch_gemm<EPI_GELU_BF16>(dev, sms, bn, split, ta, tb, ta_lo, tb_lo, ga, 0, grid); break;
      case EPI_RESID_F32: launch_gemm<EPI_RESID_F32>(dev, sms, bn, split, ta, tb, ta_lo, tb_lo, ga, 0, grid); break;
      case EPI_QKV: launch_gemm<EPI_QKV>(dev, sms, bn, split, ta, tb, ta_lo, tb_lo, ga, 0, grid); break;
      case EPI_PATCH: launch_gemm<EPI_PATCH>(dev, sms, bn, split, ta, tb, ta_lo, tb_lo, ga, 0, grid); break;
      default: throw std::runtime_error("unknown epilogue " + std::to_string(epi));
    }
    return static_cast<int>(cudaDeviceSynchronize());
  } catch (const std::exception& ex) {
    fprintf(stderr, "gemm_run: %s\n", ex.what());
    return -1;
  }
}

}  // extern "C"
