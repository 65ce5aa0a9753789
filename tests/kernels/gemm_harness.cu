// Stand-alone launcher of the tcgen05 GEMM (csrc/gemm.cuh) on caller-built inputs, for tests/test_gemm_gpu.py.
// Test-only code: the engine never links it.  All pointers are device pointers (torch tensors); the call synchronises
// and returns a cudaError_t (0 = success; -1 = a host-side failure, printed to stderr).
//
// The tensor maps, wbox(), the shared-memory attributes, the grids and the launches are literal copies of the engine's
// lines (engine.cu, allocate(): t_x / t_ctx / t_a1 / t_mid / t_patch and the K-chunk maps t_mid_c, which start at
// column c * kchunk of a row of pitch I; load_weights(): t_wqkv / t_wo / t_wi / t_wo2 / t_patch_w with wbox(bn) rows and
// t_wo2_c; launch_gemm / launch_gemm_t / launch_gemm_pair), so the kernels see exactly the operands and the launch they
// see inside a forward.  When the GEMM, its tensor maps or its launch change, this file changes with them.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <stdexcept>
#include <string>

#include "gemm.cuh"
#include "tmap.h"

using namespace mmee;

#define CUDA_OK(x)                                                                                   \
  do {                                                                                               \
    cudaError_t e_ = (x);                                                                            \
    if (e_ != cudaSuccess)                                                                           \
      throw std::runtime_error(std::string(#x) + ": " + cudaGetErrorString(e_) + " @" + std::to_string(__LINE__)); \
  } while (0)

namespace {

int wbox(int bn) { return bn == 256 ? 128 : bn; }   // engine.cu: weight TMA box rows for a GEMM family with BLOCK_N = bn

// engine.cu launch_gemm_t (the single-CTA kernel at BLOCK_N = 128); grid 0 = the engine's grid, e->sms
template <int BN, int EPI, bool SPLIT>
void launch_gemm_t(int sms, int grid, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta_lo,
                   const CUtensorMap& tb_lo, const GemmArgs& a) {
  auto kern = gemm_tc_kernel<BN, EPI, SPLIT>;
  CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmSmem<BN>::DYN_BYTES));
  kern<<<grid ? grid : sms, GEMM_THREADS, GemmSmem<BN>::DYN_BYTES>>>(ta, tb, ta_lo, tb_lo, a);
  CUDA_OK(cudaGetLastError());
}

// engine.cu launch_gemm_pair (BLOCK_N = 256, clusters of two CTAs); grid 0 = the engine's grid, e->sms & ~1
template <int EPI, bool SPLIT>
void launch_gemm_pair(int sms, int grid, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta_lo,
                      const CUtensorMap& tb_lo, const GemmArgs& a) {
  auto kern = gemm_tc_pair_kernel<EPI, SPLIT>;
  using PS = GemmPairSmemT<gemm_pair_epi_warps<EPI>()>;
  CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, PS::DYN_BYTES));
  kern<<<grid ? grid : (sms & ~1), PS::THREADS, PS::DYN_BYTES>>>(ta, tb, ta_lo, tb_lo, a);
  CUDA_OK(cudaGetLastError());
}

// engine.cu launch_gemm: in bf16 mode the low-part maps are the operands' own maps
template <int EPI>
void launch_gemm(int sms, int grid, int bn, int split, const CUtensorMap& ta, const CUtensorMap& tb,
                 const CUtensorMap& ta_lo, const CUtensorMap& tb_lo, const GemmArgs& a) {
  if (split) {
    if (bn == 256) launch_gemm_pair<EPI, true>(sms, grid, ta, tb, ta_lo, tb_lo, a);
    else launch_gemm_t<128, EPI, true>(sms, grid, ta, tb, ta_lo, tb_lo, a);
  } else {
    if (bn == 256) launch_gemm_pair<EPI, false>(sms, grid, ta, tb, ta, tb, a);
    else launch_gemm_t<128, EPI, false>(sms, grid, ta, tb, ta, tb, a);
  }
}

}  // namespace

extern "C" {

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
    // engine.cu allocate() / load_weights()
    const CUtensorMap ta = make_tmap_2d_sw128(a, a_rows, K, a_pitch, 128);
    const CUtensorMap tb = make_tmap_2d_sw128(w, N, K, w_pitch, wbox(bn));
    CUtensorMap ta_lo = ta, tb_lo = tb;
    if (split) {
      ta_lo = make_tmap_2d_sw128(a_lo, a_rows, K, a_pitch, 128);
      tb_lo = make_tmap_2d_sw128(w_lo, N, K, w_pitch, wbox(bn));
    }
    GemmArgs ga{};
    ga.m_dev = m_dev; ga.m_static = m_static; ga.N = N; ga.K = K; ga.bias = bias;
    ga.out = out; ga.out_lo = static_cast<__nv_bfloat16*>(out_lo); ga.ld_out = ld_out;
    ga.resid = static_cast<const __nv_bfloat16*>(resid); ga.resid_lo = static_cast<const __nv_bfloat16*>(resid_lo);
    ga.resid_f32 = resid_f32;
    ga.resid_y = resid_y; ga.resid_stats = static_cast<const float2*>(resid_stats); ga.resid_src = resid_src;
    ga.resid_w = resid_w; ga.resid_b = resid_b; ga.resid_prefetch = resid_prefetch;
    ga.vt = static_cast<__nv_bfloat16*>(vt); ga.vt_lo = static_cast<__nv_bfloat16*>(vt_lo); ga.qk_cols = qk_cols;
    ga.row0 = row0; ga.n_slots_dev = n_slots_dev; ga.kv_pitch = kv_pitch; ga.heads = heads;
    ga.pos = pos; ga.n_patch = n_patch; ga.n_vis = n_vis;
    switch (epi) {
      case EPI_BIAS_BF16: launch_gemm<EPI_BIAS_BF16>(sms, grid, bn, split, ta, tb, ta_lo, tb_lo, ga); break;
      case EPI_GELU_BF16: launch_gemm<EPI_GELU_BF16>(sms, grid, bn, split, ta, tb, ta_lo, tb_lo, ga); break;
      case EPI_RESID_F32: launch_gemm<EPI_RESID_F32>(sms, grid, bn, split, ta, tb, ta_lo, tb_lo, ga); break;
      case EPI_QKV: launch_gemm<EPI_QKV>(sms, grid, bn, split, ta, tb, ta_lo, tb_lo, ga); break;
      case EPI_PATCH: launch_gemm<EPI_PATCH>(sms, grid, bn, split, ta, tb, ta_lo, tb_lo, ga); break;
      default: throw std::runtime_error("unknown epilogue " + std::to_string(epi));
    }
    return static_cast<int>(cudaDeviceSynchronize());
  } catch (const std::exception& ex) {
    fprintf(stderr, "gemm_run: %s\n", ex.what());
    return -1;
  }
}

}  // extern "C"
