// libmmee: engine object + C ABI (include/mmee.h).  Orchestrates the sm_100a kernels for the reference's
// LayoutLMv3EEForSequenceClassification.forward (EE/models/LayoutLMv3.py:696-896) + exit policy
// (EE/policy.py:12-53) with on-device survivor compaction.  No CPU fallback: every compute step is a
// CUDA kernel from this directory.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <numeric>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/mmee.h"
#include "attention.cuh"
#include "embed.cuh"
#include "gemm.cuh"
#include "image.cuh"
#include "norm_exit.cuh"
#include "policy.cuh"
#include "calibrate.cuh"
#include "tmap.h"

using namespace mmee;

namespace {

thread_local std::string g_err;

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  void alloc(size_t count, bool zero = false) {
    release();
    n = count;
    if (count) {
      CUDA_OK(cudaMalloc(&p, count * sizeof(T)));
      if (zero) CUDA_OK(cudaMemset(p, 0, count * sizeof(T)));
    }
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
};

__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n, float scale) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16_rn(src[i] * scale);
}
// split-bf16 conversion of a weight: hi = bf16(v), lo = bf16(v - hi)   (fp32 engine mode)
__global__ void f32_to_bf16_split_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ hi,
                                         __nv_bfloat16* __restrict__ lo, size_t n, float scale) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) {
    const float v = src[i] * scale;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}
__global__ void init_forward_kernel(int* slot_doc, int* out_exit, int* n_dev, int* m_dev, unsigned long long* hist,
                                    int B, int seq, int n_hist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) { slot_doc[i] = i; out_exit[i] = -1; }
  if (i < n_hist) hist[i] = 0ull;
  if (i == 0) { n_dev[0] = B; m_dev[0] = B * seq; }     // dense upper bound; the row plan writes the ragged count
}
__global__ void fill_nan_kernel(float* p, size_t n) {
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i < n) p[i] = __int_as_float(0x7fc00000);
}
__global__ void hist_to_i64_kernel(const unsigned long long* h, long long* out, int n) {
  const int i = threadIdx.x;
  if (i < n) out[i] = static_cast<long long>(h[i]);
}

struct LayerW {
  DevBuf<__nv_bfloat16> wqkv, wo, wi, wo2;
  DevBuf<__nv_bfloat16> wqkv_lo, wo_lo, wi_lo, wo2_lo;      // fp32 engine mode: low parts of the split-bf16 weights
  DevBuf<float> bqkv, bo, bi, bo2, ln1_w, ln1_b, ln2_w, ln2_b;
  CUtensorMap t_wqkv, t_wo, t_wi, t_wo2;
  CUtensorMap t_wqkv_lo, t_wo_lo, t_wi_lo, t_wo2_lo;
  std::vector<CUtensorMap> t_wo2_c, t_wo2_lo_c;             // fp32 engine mode: MLP-down weight in K chunks (see kchunk)
};

struct HeadW {
  DevBuf<float> dense_w, dense_b, out_w, out_b;
  int n_out = 0;
  bool two_layer = false;
  HeadWeights view() const {
    HeadWeights h;
    h.dense_w = two_layer ? dense_w.p : nullptr;
    h.dense_b = dense_b.p;
    h.out_w = out_w.p;
    h.out_b = out_b.p;
    h.n_out = n_out;
    return h;
  }
};

}  // namespace

struct mmee_engine {
  mmee_model_desc d;
  int device = 0;
  int max_batch = 0;
  int H, L, heads, I, T, P, S, K, n_vis, n_patch, kdim_patch;
  int kv_pitch = 768, bias_pitch = 768;
  bool split = false;              // fp32 engine mode (mmee_model_desc.compute_dtype == MMEE_DTYPE_FP32): split-bf16 operands
  // ragged encoder layout (norm_exit.cuh): kept tokens per document and the row plans of two consecutive exit stages
  DevBuf<int> doc_len, kept_idx, plan_row0[2], plan_qt_slot[2], plan_n_qt[2];
  DevBuf<int4> plan_meta[2];
  bool tail16 = true;              // attention: a last key tile with <= 16 real keys runs as a 16-key tile (MMEE_NO_TAIL16=1: off)
  DevBuf<float> lte_w, slot_lte;   // learned-to-exit scorer [H] (optional) and its per-slot scores
  float lte_b = 0.f;
  int m_max = 0;            // padded row capacity of activation buffers
  int sms = 148;
  int bn_h, bn_qkv, bn_i;   // BLOCK_N per GEMM family
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;       // host path: pixel upload overlaps text embedding + bias build
  cudaEvent_t px_ready = nullptr;           // recorded on copy_stream after the pixel copy
  cudaEvent_t fwd_start = nullptr;
  bool px_async = false;                    // forward_device must wait for px_ready before touching pixels
  bool finalized = false;
  int64_t launches = 0;
  bool profiling = false;
  std::map<std::string, double> stage_ms;
  std::vector<std::pair<std::string, cudaEvent_t>> ev;

  // raw fp32 staging of weights until finalize
  std::map<std::string, std::vector<float>> raw;
  std::map<std::string, std::vector<int64_t>> raw_shape;

  // weights
  std::vector<LayerW> layers;
  DevBuf<float> word, type0, pos, x_emb, y_emb, h_emb, w_emb, ln_emb_w, ln_emb_b, ln_model_w, ln_model_b, ln_vis_w,
      ln_vis_b, cls_token, pos_embed, patch_b, w1d, wx, wy;
  DevBuf<__nv_bfloat16> patch_w, patch_w_lo;
  CUtensorMap t_patch_w, t_patch_w_lo;
  std::vector<HeadW> exit_heads;     // one per configured exit (concat first if present)
  HeadW classifier;
  DevBuf<uint8_t> lut1, lut2;
  std::vector<uint8_t> h_lut1, h_lut2;
  DevBuf<int> vis_bbox;

  // activations
  DevBuf<__nv_bfloat16> X[2], QK, VT, CTX, A1, MID, PATCH;
  DevBuf<__nv_bfloat16> Xlo[2], A1lo;       // low parts of the split-bf16 residual stream (precise_residual without y_resid)
  // y_resid (bf16 mode, H % 128 == 0): residual adds recompute LayerNorm(pre-LN sums) instead of reading (hi, lo) pairs.
  // Y2 = out-projection output (Y stays the MLP-down output the next layer's residual is recomputed from), per-row
  // (mean, rstd) of both LayerNorms, and for the post-MLP one the source row in Y (exit compaction moves rows)
  bool y_resid = false;
  DevBuf<float> Y2;
  DevBuf<float2> ln_stats1, ln_stats2;
  DevBuf<int> ln_src2;
  DevBuf<__nv_bfloat16> QKlo, VTlo, CTXlo, MIDlo, PATCHlo;   // fp32 engine mode: low parts of every other GEMM / attention operand
  DevBuf<__half> BIASlo;                    // fp32 engine mode: low part of the attention bias
  DevBuf<float> X32[2], A132;               // fp32 engine mode: the residual stream itself in fp32 (exact residual adds)
  // fp32 engine mode: the MLP-down GEMM runs in K chunks (gemm_kchunk; measured without them: 2e-5 relative error at
  // K = 3072 x 3 segments); every chunk after the first adds to the running sum Y
  int kchunk = 0, n_kchunks = 1;
  std::vector<CUtensorMap> t_mid_c, t_mid_lo_c;
  DevBuf<float> zero_bias;
  bool precise_residual = true;
  DevBuf<float> Y, VIS, POOL, POOLV, POOLT, TXT, Z, T0, T1;
  bool has_vision_exit = false, has_text_exit = false;
  DevBuf<__half> BIAS, bias_t2;
  DevBuf<float> maskadd, bias_t1, bias_tx, bias_ty;     // bias_tx / bias_ty: fp32 engine mode (bias_build_split_kernel)
  DevBuf<int> err_flags;                    // err_flags: [0] attention online-softmax guard, [1] input id / box out of range
  cudaEvent_t last_done = nullptr;          // end of the last forward: the next one (any stream) is ordered after it
  DevBuf<long long> att_trace;
  bool trace_on = false;
  int n_kv_tiles = 6;
  DevBuf<int> posid;
  CUtensorMap t_x[2], t_ctx, t_a1, t_mid, t_patch;
  CUtensorMap t_x_lo[2], t_ctx_lo, t_a1_lo, t_mid_lo, t_patch_lo;   // fp32 engine mode
  AttMaps att_maps;

  // bookkeeping (device)
  DevBuf<int> n_dev, m_dev;                 // [stages]
  DevBuf<int> slot_doc[2], slot_src;        // ping-pong slot->doc; new->old slot map
  DevBuf<int> slot_fire, out_exit;
  DevBuf<unsigned int> exit_tickets;        // exit_fused_kernel: per-group tickets + groups-done counter
  DevBuf<float> slot_logits, slot_head, slot_crit, out_logits, out_crit, all_logits, all_head, all_crit;
  DevBuf<unsigned long long> hist;
  DevBuf<long long> hist64;
  // staged inputs (host path)
  DevBuf<int64_t> in_ids, in_bbox, in_mask;
  DevBuf<float> in_px;
  // pipelined host path (mmee_forward_submit / mmee_forward_collect): two forwards in flight
  struct Slot {
    DevBuf<int64_t> ids, bbox, mask;
    DevBuf<float> px, logits, crit;
    DevBuf<int32_t> exit_index;
    DevBuf<int64_t> hist;
    cudaEvent_t small_ready = nullptr, px_ready = nullptr, done = nullptr;
    int B = 0;
    bool busy = false;
  } slots[2];
  int next_slot = 0;
  cudaEvent_t px_wait = nullptr;            // event forward_device waits on before touching pixels (px_async)
  // uint8 image preprocess (image.cuh), grow-only: packed batch of the host path, first-pass intermediate,
  // coefficient tables, and the per-call descriptors (ImageDesc[max_batch] + ImageAxis[2 max_batch]) with their pinned
  // staging.  img_done orders preprocess calls on any streams (they share this scratch).
  DevBuf<uint8_t> img_bytes, img_tmp, img_meta;
  DevBuf<int> img_kk;
  DevBuf<int2> img_bounds;
  uint8_t* img_meta_host = nullptr;
  cudaEvent_t img_meta_copied = nullptr, img_done = nullptr;
  // captured forwards (mmee_plan_create): run on the same scratch buffers, freed by mmee_destroy if still alive
  std::vector<mmee_plan*> plans;
  bool capturing = false;                   // forward_device is recording a plan: no stage events

  ~mmee_engine() {
    for (auto& sl : slots) {
      if (sl.small_ready) cudaEventDestroy(sl.small_ready);
      if (sl.px_ready) cudaEventDestroy(sl.px_ready);
      if (sl.done) cudaEventDestroy(sl.done);
    }
    for (auto& e : ev) cudaEventDestroy(e.second);
    if (stream) cudaStreamDestroy(stream);
    if (copy_stream) cudaStreamDestroy(copy_stream);
    if (px_ready) cudaEventDestroy(px_ready);
    if (last_done) cudaEventDestroy(last_done);
    if (fwd_start) cudaEventDestroy(fwd_start);
    if (img_meta_copied) cudaEventDestroy(img_meta_copied);
    if (img_done) cudaEventDestroy(img_done);
    if (img_meta_host) cudaFreeHost(img_meta_host);
  }
};

namespace {

int n_stages(const mmee_engine* e) { return e->d.n_exits + 3; }

SlotRows plan_view(mmee_engine* e, int i) {
  SlotRows r;
  r.row0 = e->plan_row0[i].p; r.meta = e->plan_meta[i].p; r.qt_slot = e->plan_qt_slot[i].p; r.n_qt_dev = e->plan_n_qt[i].p;
  return r;
}

std::vector<uint8_t> default_lut(int num_buckets, int max_distance, int n) {
  // HF relative_position_bucket (modeling_layoutlmv3.py:393-414), bidirectional: table over |rel|.
  const int nb = num_buckets / 2;
  const int max_exact = nb / 2;
  std::vector<uint8_t> lut(n);
  const float denom = static_cast<float>(log(static_cast<double>(max_distance) / max_exact));
  for (int i = 0; i < n; ++i) {
    int v;
    if (i < max_exact) {
      v = i;
    } else {
      const float q = static_cast<float>(i) / static_cast<float>(max_exact);
      const float val = logf(q) / denom * static_cast<float>(nb - max_exact);
      v = max_exact + static_cast<int>(val);
      if (v > nb - 1) v = nb - 1;
    }
    lut[i] = static_cast<uint8_t>(v);
  }
  return lut;
}

const std::vector<float>& need(mmee_engine* e, const std::string& name, std::initializer_list<int64_t> shape) {
  auto it = e->raw.find(name);
  if (it == e->raw.end()) throw std::runtime_error("missing weight: " + name);
  size_t n = 1;
  for (auto s : shape) n *= static_cast<size_t>(s);
  if (it->second.size() != n)
    throw std::runtime_error("bad size for " + name + ": got " + std::to_string(it->second.size()) + " want " +
                             std::to_string(n));
  return it->second;
}

void upload_f32(DevBuf<float>& dst, const std::vector<float>& src, float scale = 1.f) {
  dst.alloc(src.size());
  if (scale == 1.f) {
    CUDA_OK(cudaMemcpy(dst.p, src.data(), src.size() * 4, cudaMemcpyHostToDevice));
  } else {
    std::vector<float> t(src);
    for (auto& v : t) v *= scale;
    CUDA_OK(cudaMemcpy(dst.p, t.data(), t.size() * 4, cudaMemcpyHostToDevice));
  }
}

// dst[offset ...] = bf16(src * scale)
void upload_bf16(__nv_bfloat16* dst, const std::vector<float>& src, float scale = 1.f) {
  DevBuf<float> tmp;
  tmp.alloc(src.size());
  CUDA_OK(cudaMemcpy(tmp.p, src.data(), src.size() * 4, cudaMemcpyHostToDevice));
  f32_to_bf16_kernel<<<static_cast<unsigned>((src.size() + 255) / 256), 256>>>(tmp.p, dst, src.size(), scale);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaDeviceSynchronize());
}

// hi[...] = bf16(src * scale), lo[...] = bf16(src * scale - hi)
void upload_bf16_split(__nv_bfloat16* hi, __nv_bfloat16* lo, const std::vector<float>& src, float scale = 1.f) {
  DevBuf<float> tmp;
  tmp.alloc(src.size());
  CUDA_OK(cudaMemcpy(tmp.p, src.data(), src.size() * 4, cudaMemcpyHostToDevice));
  f32_to_bf16_split_kernel<<<static_cast<unsigned>((src.size() + 255) / 256), 256>>>(tmp.p, hi, lo, src.size(), scale);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaDeviceSynchronize());
}

void load_head(mmee_engine* e, HeadW& h, const std::string& prefix, int n_out) {
  const int H = e->H;
  h.n_out = n_out;
  h.two_layer = e->d.head_layers == 2;
  if (h.two_layer) {
    upload_f32(h.dense_w, need(e, prefix + ".dense.weight", {H, H}));
    upload_f32(h.dense_b, need(e, prefix + ".dense.bias", {H}));
  }
  upload_f32(h.out_w, need(e, prefix + ".out_proj.weight", {n_out, H}));
  upload_f32(h.out_b, need(e, prefix + ".out_proj.bias", {n_out}));
}

// ta_lo / tb_lo: tensor maps of the operands' low parts (fp32 engine mode: three k segments); unused in bf16 mode
template <int EPI>
void run_gemm(mmee_engine* e, int bn, const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& ta_lo,
              const CUtensorMap& tb_lo, const GemmArgs& a, cudaStream_t st) {
  launch_gemm<EPI>(e->device, e->sms, bn, e->split, ta, tb, ta_lo, tb_lo, a, st);
  e->launches++;
}

template <typename F>
void launch_nv(int H, F&& f) {   // dispatch on values-per-lane for the warp-per-row kernels
  if (H <= 128) f(std::integral_constant<int, 4>{});
  else if (H <= 256) f(std::integral_constant<int, 8>{});
  else if (H <= 768) f(std::integral_constant<int, 24>{});
  else if (H <= 1024) f(std::integral_constant<int, 32>{});
  else throw std::runtime_error("hidden size > 1024 not supported");
}

// LayerNorm of the active rows (fp32 Y -> bf16 X [+ low part, + fp32 copy]); vectorised when H is a multiple of 128.
// slot_src != nullptr: the rows are the survivors of an exit — destination slot s' (row plan `dst`) takes the rows of
// source slot slot_src[s'] (row plan `src`): the compaction costs no extra pass.
void launch_ln(mmee_engine* e, const float* Y, __nv_bfloat16* X, __nv_bfloat16* Xlo, float* X32, const float* w,
               const float* b, int B, const int* m_dev, const int* slot_src, const SlotRows& dst, const SlotRows& src,
               const int* n_dst_dev, cudaStream_t st, float2* stats_out = nullptr, int* src_out = nullptr) {
  const int H = e->H, S = e->S;
  const float eps = e->d.ln_eps;
  const int rows = B * S;
  auto vec = [&](auto nv4) {
    const int blocks = std::min((rows + 7) / 8, e->sms * 16);      // grid-stride over rows, 8 warps per block
    ln_rows_vec_kernel<decltype(nv4)::value><<<blocks, 256, 0, st>>>(Y, X, Xlo, X32, w, b, eps, H, m_dev, slot_src, dst.row0,
                                                                       src.row0, n_dst_dev, stats_out, src_out);
  };
  switch (H % 128 == 0 ? H / 128 : 0) {
    case 1: vec(std::integral_constant<int, 1>{}); break;
    case 2: vec(std::integral_constant<int, 2>{}); break;
    case 3: vec(std::integral_constant<int, 3>{}); break;
    case 4: vec(std::integral_constant<int, 4>{}); break;
    case 5: vec(std::integral_constant<int, 5>{}); break;
    case 6: vec(std::integral_constant<int, 6>{}); break;
    case 7: vec(std::integral_constant<int, 7>{}); break;
    case 8: vec(std::integral_constant<int, 8>{}); break;
    default:
      if (stats_out) throw std::runtime_error("residual statistics need the vectorised LayerNorm (H % 128 == 0)");
      launch_nv(H, [&](auto nv) {
        ln_rows_kernel<decltype(nv)::value><<<(rows + 7) / 8, 256, 0, st>>>(Y, X, Xlo, X32, w, b, eps, H, m_dev, slot_src,
                                                                            dst.row0, src.row0, n_dst_dev);
      });
  }
  CUDA_OK(cudaGetLastError());
}

void mark(mmee_engine* e, const char* name, cudaStream_t st) {
  if (!e->profiling || e->capturing) return;
  cudaEvent_t evn;
  CUDA_OK(cudaEventCreate(&evn));
  CUDA_OK(cudaEventRecord(evn, st));
  e->ev.emplace_back(name, evn);
}

void finalize(mmee_engine* e) {
  const mmee_model_desc& d = e->d;
  const int H = e->H, I = e->I, h = e->heads;
  CUDA_OK(cudaSetDevice(e->device));
  const std::string p = "layoutlmv3.";
  const std::string em = p + "embeddings.";
  upload_f32(e->word, need(e, em + "word_embeddings.weight", {d.vocab, H}));
  {
    const auto& tt = e->raw.at(em + "token_type_embeddings.weight");
    if (tt.size() < static_cast<size_t>(H)) throw std::runtime_error("token_type_embeddings too small");
    std::vector<float> row0(tt.begin(), tt.begin() + H);
    upload_f32(e->type0, row0);
  }
  upload_f32(e->pos, need(e, em + "position_embeddings.weight", {d.max_pos, H}));
  upload_f32(e->x_emb, need(e, em + "x_position_embeddings.weight", {d.max_2d, d.coord}));
  upload_f32(e->y_emb, need(e, em + "y_position_embeddings.weight", {d.max_2d, d.coord}));
  upload_f32(e->h_emb, need(e, em + "h_position_embeddings.weight", {d.max_2d, d.shape}));
  upload_f32(e->w_emb, need(e, em + "w_position_embeddings.weight", {d.max_2d, d.shape}));
  upload_f32(e->ln_emb_w, need(e, em + "LayerNorm.weight", {H}));
  upload_f32(e->ln_emb_b, need(e, em + "LayerNorm.bias", {H}));
  upload_f32(e->ln_model_w, need(e, p + "LayerNorm.weight", {H}));
  upload_f32(e->ln_model_b, need(e, p + "LayerNorm.bias", {H}));
  upload_f32(e->ln_vis_w, need(e, p + "norm.weight", {H}));
  upload_f32(e->ln_vis_b, need(e, p + "norm.bias", {H}));
  upload_f32(e->cls_token, need(e, p + "cls_token", {H}));
  upload_f32(e->pos_embed, need(e, p + "pos_embed", {e->n_vis, H}));
  upload_f32(e->patch_b, need(e, p + "patch_embed.proj.bias", {H}));
  const bool split = e->split;
  // one GEMM weight: bf16 (bf16 mode) or the split pair (fp32 mode)
  auto upload_w = [&](DevBuf<__nv_bfloat16>& hi, DevBuf<__nv_bfloat16>& lo, size_t offset, size_t total,
                      const std::vector<float>& src, float scale = 1.f) {
    if (!hi.p) hi.alloc(total);
    if (split && !lo.p) lo.alloc(total);
    if (split) upload_bf16_split(hi.p + offset, lo.p + offset, src, scale);
    else upload_bf16(hi.p + offset, src, scale);
  };
  upload_w(e->patch_w, e->patch_w_lo, 0, static_cast<size_t>(H) * e->kdim_patch,
           need(e, p + "patch_embed.proj.weight", {H, e->kdim_patch}));
  upload_f32(e->w1d, need(e, p + "encoder.rel_pos_bias.weight", {h, d.rel_bins}));
  upload_f32(e->wx, need(e, p + "encoder.rel_pos_x_bias.weight", {h, d.rel2d_bins}));
  upload_f32(e->wy, need(e, p + "encoder.rel_pos_y_bias.weight", {h, d.rel2d_bins}));

  // Q carries log2(e)/sqrt(d): the attention softmax runs in the log2 domain (exp2 without a per-element multiply)
  const float qscale = 1.4426950408889634f / sqrtf(static_cast<float>(H / h));
  {
    // attention-bias tables in the log2 domain (bias_build_kernel): T1[b1][head] = W1d * c (fp32),
    // T2[bx][by][head] = fp16((Wx + Wy) * c), c = log2(e)/sqrt(d)
    const auto& t1 = need(e, p + "encoder.rel_pos_bias.weight", {h, d.rel_bins});
    const auto& tx = need(e, p + "encoder.rel_pos_x_bias.weight", {h, d.rel2d_bins});
    const auto& ty = need(e, p + "encoder.rel_pos_y_bias.weight", {h, d.rel2d_bins});
    if (h % 2) throw std::runtime_error("attention heads must be even");
    const int t2p = bias_table_pitch(h);         // table row pitch (elements)
    std::vector<float> T1(static_cast<size_t>(d.rel_bins) * t2p, 0.f);
    for (int b1 = 0; b1 < d.rel_bins; ++b1)
      for (int hh = 0; hh < h; ++hh) T1[static_cast<size_t>(b1) * t2p + hh] = t1[static_cast<size_t>(hh) * d.rel_bins + b1] * qscale;
    std::vector<__half> T2(static_cast<size_t>(d.rel2d_bins) * d.rel2d_bins * t2p, __float2half_rn(0.f));
    for (int bx = 0; bx < d.rel2d_bins; ++bx)
      for (int by = 0; by < d.rel2d_bins; ++by)
        for (int hh = 0; hh < h; ++hh)
          T2[(static_cast<size_t>(bx) * d.rel2d_bins + by) * t2p + hh] = __float2half_rn(
              (tx[static_cast<size_t>(hh) * d.rel2d_bins + bx] + ty[static_cast<size_t>(hh) * d.rel2d_bins + by]) * qscale);
    upload_f32(e->bias_t1, T1);
    if (e->split) {                                // fp32 tables for the split bias builder
      std::vector<float> TX(static_cast<size_t>(d.rel2d_bins) * t2p, 0.f), TY(TX.size(), 0.f);
      for (int b2 = 0; b2 < d.rel2d_bins; ++b2)
        for (int hh = 0; hh < h; ++hh) {
          TX[static_cast<size_t>(b2) * t2p + hh] = tx[static_cast<size_t>(hh) * d.rel2d_bins + b2] * qscale;
          TY[static_cast<size_t>(b2) * t2p + hh] = ty[static_cast<size_t>(hh) * d.rel2d_bins + b2] * qscale;
        }
      upload_f32(e->bias_tx, TX);
      upload_f32(e->bias_ty, TY);
    }
    e->bias_t2.alloc(T2.size());
    CUDA_OK(cudaMemcpy(e->bias_t2.p, T2.data(), T2.size() * 2, cudaMemcpyHostToDevice));
  }
  e->layers.resize(e->L);
  for (int i = 0; i < e->L; ++i) {
    LayerW& w = e->layers[i];
    const std::string lp = p + "encoder.layer." + std::to_string(i) + ".";
    const size_t hh = static_cast<size_t>(H) * H;
    upload_w(w.wqkv, w.wqkv_lo, 0, 3 * hh, need(e, lp + "attention.self.query.weight", {H, H}), qscale);
    upload_w(w.wqkv, w.wqkv_lo, hh, 3 * hh, need(e, lp + "attention.self.key.weight", {H, H}));
    upload_w(w.wqkv, w.wqkv_lo, 2 * hh, 3 * hh, need(e, lp + "attention.self.value.weight", {H, H}));
    {
      std::vector<float> b(3 * H);
      const auto& bq = need(e, lp + "attention.self.query.bias", {H});
      const auto& bk = need(e, lp + "attention.self.key.bias", {H});
      const auto& bv = need(e, lp + "attention.self.value.bias", {H});
      for (int j = 0; j < H; ++j) { b[j] = bq[j] * qscale; b[H + j] = bk[j]; b[2 * H + j] = bv[j]; }
      upload_f32(w.bqkv, b);
    }
    upload_w(w.wo, w.wo_lo, 0, hh, need(e, lp + "attention.output.dense.weight", {H, H}));
    upload_f32(w.bo, need(e, lp + "attention.output.dense.bias", {H}));
    upload_f32(w.ln1_w, need(e, lp + "attention.output.LayerNorm.weight", {H}));
    upload_f32(w.ln1_b, need(e, lp + "attention.output.LayerNorm.bias", {H}));
    upload_w(w.wi, w.wi_lo, 0, static_cast<size_t>(I) * H, need(e, lp + "intermediate.dense.weight", {I, H}));
    upload_f32(w.bi, need(e, lp + "intermediate.dense.bias", {I}));
    upload_w(w.wo2, w.wo2_lo, 0, static_cast<size_t>(H) * I, need(e, lp + "output.dense.weight", {H, I}));
    upload_f32(w.bo2, need(e, lp + "output.dense.bias", {H}));
    upload_f32(w.ln2_w, need(e, lp + "output.LayerNorm.weight", {H}));
    upload_f32(w.ln2_b, need(e, lp + "output.LayerNorm.bias", {H}));
    w.t_wqkv = gemm_w_map(w.wqkv.p, 3 * H, H, H, e->bn_qkv);
    w.t_wo = gemm_w_map(w.wo.p, H, H, H, e->bn_h);
    w.t_wi = gemm_w_map(w.wi.p, I, H, H, e->bn_i);
    w.t_wo2 = gemm_w_map(w.wo2.p, H, I, I, e->bn_h);
    if (split) {
      w.t_wqkv_lo = gemm_w_map(w.wqkv_lo.p, 3 * H, H, H, e->bn_qkv);
      w.t_wo_lo = gemm_w_map(w.wo_lo.p, H, H, H, e->bn_h);
      w.t_wi_lo = gemm_w_map(w.wi_lo.p, I, H, H, e->bn_i);
      w.t_wo2_lo = gemm_w_map(w.wo2_lo.p, H, I, I, e->bn_h);
      for (int c = 0; c < e->n_kchunks; ++c) {
        w.t_wo2_c.push_back(gemm_w_map(w.wo2.p, H, e->kchunk, I, e->bn_h, static_cast<size_t>(c) * e->kchunk));
        w.t_wo2_lo_c.push_back(gemm_w_map(w.wo2_lo.p, H, e->kchunk, I, e->bn_h, static_cast<size_t>(c) * e->kchunk));
      }
    }
  }
  e->t_patch_w = gemm_w_map(e->patch_w.p, H, e->kdim_patch, e->kdim_patch, e->bn_h);
  if (split) e->t_patch_w_lo = gemm_w_map(e->patch_w_lo.p, H, e->kdim_patch, e->kdim_patch, e->bn_h);

  const int n_head_out = d.head_kind == 0 ? d.n_labels : 2;
  e->exit_heads.resize(d.n_exits);
  int k_enc = 0;
  for (int x = 0; x < d.n_exits; ++x) {
    if (d.exit_after_layer[x] == MMEE_EXIT_VISION_AVG) load_head(e, e->exit_heads[x], p + "vision_exit_embeddings", n_head_out);
    else if (d.exit_after_layer[x] == MMEE_EXIT_TEXT_AVG) load_head(e, e->exit_heads[x], p + "text_exit_embeddings", n_head_out);
    else if (d.exit_after_layer[x] == 0) load_head(e, e->exit_heads[x], p + "concat_exit_embeddings", n_head_out);
    else load_head(e, e->exit_heads[x], p + "encoder.early_exits." + std::to_string(k_enc++), n_head_out);
  }
  load_head(e, e->classifier, "classifier", d.n_labels);
  e->classifier.two_layer = true;   // HF ClassificationHead always has dense + out_proj (HF:798-822)
  if (!e->classifier.dense_w.p) {
    upload_f32(e->classifier.dense_w, need(e, "classifier.dense.weight", {H, H}));
    upload_f32(e->classifier.dense_b, need(e, "classifier.dense.bias", {H}));
  }

  // optional learned-to-exit scorer (EE/models/LayoutLMv3.py:142-149): Linear(H, 1); needed for criterion 2 only
  if (e->raw.count(p + "encoder.lte_classifier.weight")) {
    upload_f32(e->lte_w, need(e, p + "encoder.lte_classifier.weight", {1, H}));
    e->lte_b = need(e, p + "encoder.lte_classifier.bias", {1})[0];
  }

  if (e->h_lut1.empty()) e->h_lut1 = default_lut(d.rel_bins, d.max_rel, 1024);
  if (e->h_lut2.empty()) e->h_lut2 = default_lut(d.rel2d_bins, d.max_rel2d, 1024);
  e->lut1.alloc(e->h_lut1.size());
  e->lut2.alloc(e->h_lut2.size());
  CUDA_OK(cudaMemcpy(e->lut1.p, e->h_lut1.data(), e->h_lut1.size(), cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(e->lut2.p, e->h_lut2.data(), e->h_lut2.size(), cudaMemcpyHostToDevice));

  // visual token boxes (HF:576-602): CLS [1,1,999,999]; grid edges trunc(1000*k/n)
  {
    const int ns = d.image / d.patch;
    std::vector<int> vb(static_cast<size_t>(e->n_vis) * 4);
    vb[0] = 1; vb[1] = 1; vb[2] = 999; vb[3] = 999;
    for (int r = 0; r < ns; ++r)
      for (int c = 0; c < ns; ++c) {
        int* b = &vb[static_cast<size_t>(1 + r * ns + c) * 4];
        b[0] = 1000 * c / ns; b[1] = 1000 * r / ns; b[2] = 1000 * (c + 1) / ns; b[3] = 1000 * (r + 1) / ns;
      }
    e->vis_bbox.alloc(vb.size());
    CUDA_OK(cudaMemcpy(e->vis_bbox.p, vb.data(), vb.size() * 4, cudaMemcpyHostToDevice));
  }
  e->raw.clear();
  e->raw_shape.clear();
  e->finalized = true;
}

void allocate(mmee_engine* e) {
  const int B = e->max_batch, S = e->S, H = e->H, I = e->I, heads = e->heads;
  e->m_max = ((B * S + 255) / 256) * 256 + 128;
  const size_t M = e->m_max;
  for (int i = 0; i < 2; ++i) e->X[i].alloc(M * H, true);
  e->QK.alloc(M * 2 * H, true);
  e->VT.alloc(static_cast<size_t>(B) * heads * 64 * e->kv_pitch, true);
  e->CTX.alloc(M * H, true);
  e->A1.alloc(M * H, true);
  if (e->y_resid) {
    e->Y2.alloc(M * H, true); e->ln_stats1.alloc(M, true); e->ln_stats2.alloc(M, true); e->ln_src2.alloc(M, true);
  } else if (e->precise_residual) {
    e->Xlo[0].alloc(M * H, true); e->Xlo[1].alloc(M * H, true); e->A1lo.alloc(M * H, true);
  }
  if (e->split) {
    e->QKlo.alloc(M * 2 * H, true);
    e->VTlo.alloc(static_cast<size_t>(B) * heads * 64 * e->kv_pitch, true);
    e->CTXlo.alloc(M * H, true);
    e->MIDlo.alloc(M * I, true);
    e->X32[0].alloc(M * H, true); e->X32[1].alloc(M * H, true); e->A132.alloc(M * H, true);
  }
  e->MID.alloc(M * I, true);
  e->Y.alloc(M * H, true);
  const size_t mp = (static_cast<size_t>(B) * e->n_patch + 255) / 256 * 256 + 128;
  e->PATCH.alloc(mp * e->kdim_patch, true);
  if (e->split) e->PATCHlo.alloc(mp * e->kdim_patch, true);
  e->VIS.alloc(static_cast<size_t>(B) * e->n_vis * H, true);
  e->POOL.alloc(static_cast<size_t>(B) * H, true);
  for (int x = 0; x < e->d.n_exits; ++x) {
    if (e->d.exit_after_layer[x] == MMEE_EXIT_VISION_AVG) e->has_vision_exit = true;
    if (e->d.exit_after_layer[x] == MMEE_EXIT_TEXT_AVG) e->has_text_exit = true;
  }
  if (e->has_vision_exit) e->POOLV.alloc(static_cast<size_t>(B) * H, true);
  if (e->has_text_exit) e->POOLT.alloc(static_cast<size_t>(B) * H, true);
  if (e->has_vision_exit || e->has_text_exit)            // text embeddings before the model LayerNorm (survivors finish later)
    e->TXT.alloc(static_cast<size_t>(B) * std::max(e->T, 1) * H, true);
  e->Z.alloc(static_cast<size_t>(B) * H, true);
  e->T0.alloc(static_cast<size_t>(B) * H, true);
  e->T1.alloc(static_cast<size_t>(B) * H, true);
  e->BIAS.alloc(static_cast<size_t>(B) * heads * S * e->bias_pitch + 64 * 1024, true);   // 12.3 MB / base document
  if (e->split) e->BIASlo.alloc(static_cast<size_t>(B) * heads * S * e->bias_pitch + 64 * 1024, true);
  e->posid.alloc(static_cast<size_t>(B) * e->T);

  e->t_x[0] = gemm_a_map(e->X[0].p, M, H, H);
  e->t_x[1] = gemm_a_map(e->X[1].p, M, H, H);
  e->att_maps = attention_maps(e->QK.p, e->QKlo.p, e->VT.p, e->VTlo.p, e->BIAS.p, e->BIASlo.p, M, H, heads, S, B,
                               e->kv_pitch, e->bias_pitch, e->split);
  e->n_kv_tiles = (S + ATT_BKV - 1) / ATT_BKV;
  if (e->n_kv_tiles > ATT_MAX_KV_TILES) throw std::runtime_error("too many key tiles");
  e->maskadd.alloc(static_cast<size_t>(B) * e->kv_pitch, true);
  e->err_flags.alloc(2, true);
  e->doc_len.alloc(B, true);
  e->kept_idx.alloc(static_cast<size_t>(B) * std::max(e->T, 1), true);
  const int max_qt = (S + ATT_BQ - 1) / ATT_BQ;
  for (int i = 0; i < 2; ++i) {
    e->plan_row0[i].alloc(B + 1, true);
    e->plan_meta[i].alloc(B, true);
    e->plan_qt_slot[i].alloc(static_cast<size_t>(B) * max_qt, true);
    e->plan_n_qt[i].alloc(1, true);
  }
  e->att_trace.alloc(4096, true);
  e->t_ctx = gemm_a_map(e->CTX.p, M, H, H);
  e->t_a1 = gemm_a_map(e->A1.p, M, H, H);
  e->t_mid = gemm_a_map(e->MID.p, M, I, I);
  e->t_patch = gemm_a_map(e->PATCH.p, mp, e->kdim_patch, e->kdim_patch);
  if (e->split) {
    e->t_x_lo[0] = gemm_a_map(e->Xlo[0].p, M, H, H);
    e->t_x_lo[1] = gemm_a_map(e->Xlo[1].p, M, H, H);
    e->t_ctx_lo = gemm_a_map(e->CTXlo.p, M, H, H);
    e->t_a1_lo = gemm_a_map(e->A1lo.p, M, H, H);
    e->t_mid_lo = gemm_a_map(e->MIDlo.p, M, I, I);
    e->t_patch_lo = gemm_a_map(e->PATCHlo.p, mp, e->kdim_patch, e->kdim_patch);
    e->kchunk = gemm_kchunk(I);
    e->n_kchunks = I / e->kchunk;
    for (int c = 0; c < e->n_kchunks; ++c) {
      e->t_mid_c.push_back(gemm_a_map(e->MID.p, M, e->kchunk, I, static_cast<size_t>(c) * e->kchunk));
      e->t_mid_lo_c.push_back(gemm_a_map(e->MIDlo.p, M, e->kchunk, I, static_cast<size_t>(c) * e->kchunk));
    }
    e->zero_bias.alloc(H, true);
  }

  const int st = n_stages(e);
  e->n_dev.alloc(st, true);
  e->m_dev.alloc(st, true);
  e->slot_doc[0].alloc(B);
  e->slot_doc[1].alloc(B);
  e->slot_src.alloc(B);
  e->slot_fire.alloc(B);
  e->exit_tickets.alloc((B + EXF_DOCS - 1) / EXF_DOCS + 1, true);
  e->out_exit.alloc(B);
  const int K = e->K, E1 = e->d.n_exits + 1;
  e->slot_logits.alloc(static_cast<size_t>(B) * K);
  e->slot_head.alloc(static_cast<size_t>(B) * K);
  e->slot_crit.alloc(B);
  e->out_logits.alloc(static_cast<size_t>(B) * K);
  e->out_crit.alloc(B);
  e->all_logits.alloc(static_cast<size_t>(E1) * B * K);
  e->all_head.alloc(static_cast<size_t>(E1) * B * K);
  e->all_crit.alloc(static_cast<size_t>(E1) * B);
  e->hist.alloc(E1, true);
  e->slot_lte.alloc(B, true);
  e->hist64.alloc(E1, true);
}

// ------------------------------------------------------------------------------------------------ forward
// Effective threshold and 1/T of exit x (x = n_exits: the final classifier) under `pol`: what exit_fused_kernel
// compares against, as launch arguments (eager forwards) or uploaded before every run of a plan.
void exit_policy(const mmee_engine* e, const mmee_policy* pol, int x, float* threshold, float* inv_temp) {
  const mmee_model_desc& d = e->d;
  const bool is_final = x == d.n_exits;
  const float Te = pol->temperatures ? pol->temperatures[x] : 1.f;
  *inv_temp = 1.0f / Te;
  *threshold = is_final ? 0.f : pol->thresholds[x];
  if (pol->criterion == MMEE_CRIT_LTE && !is_final) {
    // the reference raises EarlyExitException only inside the encoder, at layer i + 1 < num_layers where
    // num_layers = len(exit_encoder_layers) (EE/models/LayoutLMv3.py:139, 250-268); other exits are scored, never taken
    int n_enc = 0;
    for (int j = 0; j < d.n_exits; ++j) n_enc += d.exit_after_layer[j] > 0 ? 1 : 0;
    const int code = d.exit_after_layer[x];
    if (!(code > 0 && code < n_enc)) *threshold = -INFINITY;
  }
}

// Capturing mode of forward_device (mmee_plan_create): the same launch sequence is recorded into a CUDA graph.  In
// early-exit mode everything after an exit is captured into the body of an IF node whose condition the exit kernel
// sets to "someone survived", so the IF nodes nest one per exit and the deeper layers are not launched at all once
// every document has left.
struct Capture {
  const float* policy_dev = nullptr;   // [2 (E+1)] {threshold, 1/T} per exit, uploaded before every run
  bool skip_tail = false;              // early-exit mode
  cudaStream_t root = nullptr;         // captures the plan's graph
  cudaStream_t side[2] = {};           // capture the body of the innermost IF node (alternating)
  int depth = 0;                       // IF nodes opened so far
};

cudaGraph_t capturing_graph(cudaStream_t st, const cudaGraphNode_t** deps = nullptr, size_t* n_deps = nullptr) {
  cudaStreamCaptureStatus status;
  cudaGraph_t g = nullptr;
  CUDA_OK(cudaStreamGetCaptureInfo(st, &status, nullptr, &g, deps, n_deps));
  if (status != cudaStreamCaptureStatusActive) throw std::runtime_error("forward plan: stream capture is not active");
  return g;
}

// condition of the next IF node, created in the graph being captured on `st` (where its node will be added)
cudaGraphConditionalHandle capture_if_handle(cudaStream_t st) {
  cudaGraphConditionalHandle h;
  CUDA_OK(cudaGraphConditionalHandleCreate(&h, capturing_graph(st), 0, cudaGraphCondAssignDefault));
  return h;
}

// adds an IF node on `h` after the work captured so far on `st` and returns the stream that captures its body
cudaStream_t capture_open_if(Capture* cap, cudaStream_t st, cudaGraphConditionalHandle h) {
  const cudaGraphNode_t* deps = nullptr;
  size_t n_deps = 0;
  cudaGraph_t g = capturing_graph(st, &deps, &n_deps);
  cudaGraphNodeParams np{};
  np.type = cudaGraphNodeTypeConditional;
  np.conditional.handle = h;
  np.conditional.type = cudaGraphCondTypeIf;
  np.conditional.size = 1;
  cudaGraphNode_t node;
  CUDA_OK(cudaGraphAddNode(&node, g, deps, n_deps, &np));
  // work captured on `st` from here on (the root stream only: the end of the forward) follows the IF node
  CUDA_OK(cudaStreamUpdateCaptureDependencies(st, &node, 1, cudaStreamSetCaptureDependencies));
  cudaStream_t body = cap->side[cap->depth & 1];
  CUDA_OK(cudaStreamBeginCaptureToGraph(body, np.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                        cudaStreamCaptureModeThreadLocal));
  if (st != cap->root) {                   // nothing else goes into an enclosing body
    cudaGraph_t done = nullptr;
    CUDA_OK(cudaStreamEndCapture(st, &done));
  }
  cap->depth += 1;
  return body;
}

void forward_device(mmee_engine* e, int B, const int64_t* ids, const int64_t* bbox, const int64_t* mask,
                    const float* px, const mmee_policy* pol, const mmee_outputs* out, cudaStream_t st,
                    Capture* cap = nullptr) {
  if (!e->finalized) throw std::runtime_error("weights not finalized");
  if (B < 1 || B > e->max_batch) throw std::runtime_error("batch out of range");
  if (!pol || (e->d.n_exits > 0 && !pol->thresholds)) throw std::runtime_error("policy/thresholds missing");
  if (!out || !out->logits || !out->exit_index) throw std::runtime_error("outputs missing");
  if (pol->criterion < 0 || pol->criterion > 2) throw std::runtime_error("criterion must be 0, 1 or 2");
  if (pol->criterion == MMEE_CRIT_LTE && !e->lte_w.p)
    throw std::runtime_error("criterion LTE needs the weights layoutlmv3.encoder.lte_classifier.{weight,bias}");
  const mmee_model_desc& d = e->d;
  const int H = e->H, S = e->S, T = e->T, K = e->K, heads = e->heads, I = e->I;
  const int E = d.n_exits, E1 = E + 1;
  const bool leave = pol->mode == 1;
  const bool gate = d.head_kind == 1;
  e->launches = 0;
  if (!cap && (!e->profiling || e->ev.size() > 100000)) {  // profiling: the events of every forward since the last
    for (auto& x : e->ev) cudaEventDestroy(x.second);      // collect are kept and folded together (stage averages)
    e->ev.clear();
  }
  // the engine has ONE set of scratch buffers: a forward on any stream is ordered after the previous forward (recorded
  // at its end below), whichever stream that one ran on (a plan run does the same around its graph launch)
  if (!cap) CUDA_OK(cudaStreamWaitEvent(st, e->last_done, 0));
  mark(e, "start", st);
  if (cap) {   // stages whose exit kernel a run skips read -1 (mmee_debug_read "NDEV")
    CUDA_OK(cudaMemsetAsync(e->n_dev.p + 1, 0xff, (e->n_dev.n - 1) * sizeof(int), st));
  }

  init_forward_kernel<<<(std::max(B, E1) + 255) / 256, 256, 0, st>>>(e->slot_doc[0].p, e->out_exit.p, e->n_dev.p,
                                                                       e->m_dev.p, e->hist.p, B, S, E1);
  e->launches++;
  const bool want_all = out->all_exit_logits || out->all_head_logits || out->all_criteria;
  if (want_all) {
    const size_t n1 = static_cast<size_t>(E1) * B * K, n2 = static_cast<size_t>(E1) * B;
    fill_nan_kernel<<<static_cast<unsigned>((n1 + 255) / 256), 256, 0, st>>>(e->all_logits.p, n1);
    fill_nan_kernel<<<static_cast<unsigned>((n1 + 255) / 256), 256, 0, st>>>(e->all_head.p, n1);
    fill_nan_kernel<<<static_cast<unsigned>((n2 + 255) / 256), 256, 0, st>>>(e->all_crit.p, n2);
    e->launches += 3;
  }

  // ---- bookkeeping of the exit stages
  int stage = 0;       // index into n_dev / m_dev
  int rp = 0;          // row plan (plan_view) of the current stage; every compaction writes the other one
  int cur = 0;         // X buffer holding the current layer input
  int sd = 0;          // slot_doc ping-pong index
  int exit_no = 0;     // next exit to evaluate
  const bool split = e->split;                    // fp32 engine mode: every GEMM operand carries a low part
  bool x_lo_valid = split;   // X[cur] has a low part (bf16 mode: not for the embedding output, a single bf16 rounding)

  auto run_exit = [&](const float* rows, size_t row_stride, const float* ln_w, const float* ln_b,
                      const HeadW& head, bool is_final, const int* rows_slot_src, const int* row_off = nullptr) {
    // one fused launch: CLS rows (+LN) -> dense/tanh -> out_proj, temperature, criterion, threshold -> compaction
    const bool use_cls = gate && !is_final;               // class logits = classifier(CLS_j) ("gated logits")
    const bool need_head = !use_cls || want_all;          // the 2-way gate output is only an API output
    ExitFusedArgs xa{};
    xa.rows = rows; xa.row_stride = row_stride; xa.row_off = row_off; xa.slot_src = rows_slot_src; xa.ln_w = ln_w; xa.ln_b = ln_b;
    xa.ln_eps = d.ln_eps; xa.H = H; xa.n_active_dev = e->n_dev.p + stage;
    int jobs = 0;
    xa.head_src = -1; xa.cls_src = -1;
    if (need_head) {
      if (head.two_layer) {
        xa.w[jobs] = head.dense_w.p; xa.b[jobs] = head.dense_b.p; xa.T[jobs] = e->T0.p; xa.head_src = jobs; ++jobs;
      } else {
        xa.head_src = 2;
      }
    }
    if (use_cls) {
      xa.w[jobs] = e->classifier.dense_w.p; xa.b[jobs] = e->classifier.dense_b.p; xa.T[jobs] = e->T1.p; xa.cls_src = jobs; ++jobs;
    }
    xa.jobs = jobs;
    xa.head = head.view();
    if (!need_head) xa.head.out_w = nullptr;
    xa.cls = e->classifier.view();
    xa.gate_mode = use_cls ? 1 : 0;
    xa.n_labels = K;
    xa.criterion = pol->criterion;
    exit_policy(e, pol, exit_no, &xa.threshold, &xa.inv_temp);
    if (cap) xa.policy = cap->policy_dev + 2 * exit_no;
    xa.force = is_final ? 1 : 0;
    if (pol->criterion == MMEE_CRIT_LTE) {
      xa.lte_w = e->lte_w.p; xa.lte_b = e->lte_b; xa.slot_lte = e->slot_lte.p;
    }
    const bool open_if = cap && cap->skip_tail && !is_final;
    if (open_if) { xa.cond = capture_if_handle(st); xa.set_cond = 1; }
    xa.slot_logits = e->slot_logits.p; xa.slot_head = e->slot_head.p; xa.slot_crit = e->slot_crit.p;
    xa.slot_fire = e->slot_fire.p;
    xa.group_ticket = e->exit_tickets.p; xa.groups_done = e->exit_tickets.p + (e->max_batch + EXF_DOCS - 1) / EXF_DOCS;
    CompactArgs& ca = xa.compact;
    ca.n_active_dev = e->n_dev.p + stage; ca.n_next_dev = e->n_dev.p + stage + 1; ca.m_next_dev = e->m_dev.p + stage + 1;
    ca.seq = S; ca.slot_doc = e->slot_doc[sd].p; ca.next_slot_doc = e->slot_doc[sd ^ 1].p;
    ca.next_slot_src = e->slot_src.p; ca.slot_fire = e->slot_fire.p; ca.slot_logits = e->slot_logits.p;
    ca.slot_head = e->slot_head.p; ca.slot_crit = e->slot_crit.p; ca.K = K;
    ca.n_head = need_head ? head.n_out : 0;
    ca.exit_index = exit_no; ca.leave = (leave || is_final) ? 1 : 0;
    ca.out_logits = e->out_logits.p; ca.out_crit = e->out_crit.p; ca.out_exit = e->out_exit.p;
    ca.all_logits = want_all ? e->all_logits.p : nullptr; ca.all_head = want_all ? e->all_head.p : nullptr;
    ca.all_crit = want_all ? e->all_crit.p : nullptr; ca.B = B; ca.n_head_max = K; ca.hist = e->hist.p;
    ca.doc_len = e->doc_len.p; ca.next_rows = plan_view(e, rp ^ 1); ca.q_rows = ATT_BQ;
    const size_t smem = exit_fused_smem(H);
    static bool configured_dev[64] = {};
    bool& configured = configured_dev[e->device & 63];   // the attribute is per device
    if (!configured) {
      CUDA_OK(cudaFuncSetAttribute(exit_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
      configured = true;
    }
    const dim3 grid(jobs ? H / EXF_FEATS : 1, (B + EXF_DOCS - 1) / EXF_DOCS, jobs ? jobs : 1);
    exit_fused_kernel<<<grid, EXF_THREADS, smem, st>>>(xa);
    CUDA_OK(cudaGetLastError());
    e->launches++;
    if (open_if) st = capture_open_if(cap, st, xa.cond);   // the rest of the forward runs only if someone survived
    stage += 1; sd ^= 1; rp ^= 1; exit_no += 1;
  };

  // ---- embeddings
  EmbedWeights ew;
  ew.word = e->word.p; ew.type0 = e->type0.p; ew.pos = e->pos.p; ew.x_emb = e->x_emb.p; ew.y_emb = e->y_emb.p;
  ew.h_emb = e->h_emb.p; ew.w_emb = e->w_emb.p; ew.ln_emb_w = e->ln_emb_w.p; ew.ln_emb_b = e->ln_emb_b.p;
  ew.ln_model_w = e->ln_model_w.p; ew.ln_model_b = e->ln_model_b.p; ew.ln_vis_w = e->ln_vis_w.p;
  ew.ln_vis_b = e->ln_vis_b.p; ew.cls_token = e->cls_token.p; ew.pos_embed = e->pos_embed.p;
  // residual-stream outputs of the embedding stage: bf16 row (+ low part and fp32 copy in the fp32 engine mode)
  auto xout = [&](int buf) { return RowOut{e->X[buf].p, split ? e->Xlo[buf].p : nullptr, split ? e->X32[buf].p : nullptr}; };

  // text embeddings of the documents in `slots` (nullptr: all B): X rows (fused, model LayerNorm applied) and / or the
  // rows before the model LayerNorm (`pre`, indexed by slot)
  auto text_embed = [&](const int* slots, const int* n_act, RowOut xo, float* pre) {
    TextEmbedArgs ta{};
    ta.ids = ids; ta.bbox = bbox; ta.posid = e->posid.p; ta.X = xo.X; ta.Xlo = xo.Xlo; ta.X32 = xo.X32; ta.pre = pre; ta.slot_doc = slots;
    ta.n_active_dev = n_act; ta.n_docs = B; ta.n_text = T; ta.seq = S; ta.H = H; ta.coord = d.coord; ta.shape = d.shape;
    ta.vocab = d.vocab; ta.max_2d = d.max_2d; ta.eps = d.ln_eps; ta.err_flag = e->err_flags.p + 1;
    const int blocks = (B * T + 7) / 8;
    auto scalar = [&]() {
      launch_nv(H, [&](auto nv) { text_embed_kernel<decltype(nv)::value><<<blocks, 256, 0, st>>>(ta, ew); });
    };
    if (H % 128 == 0 && d.coord % 4 == 0 && d.shape % 4 == 0) {
      switch (H / 128) {
        case 1: text_embed_vec_kernel<1><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 2: text_embed_vec_kernel<2><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 3: text_embed_vec_kernel<3><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 4: text_embed_vec_kernel<4><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 5: text_embed_vec_kernel<5><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 6: text_embed_vec_kernel<6><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 7: text_embed_vec_kernel<7><<<blocks, 256, 0, st>>>(ta, ew); break;
        case 8: text_embed_vec_kernel<8><<<blocks, 256, 0, st>>>(ta, ew); break;
        default: scalar();
      }
    } else {
      scalar();
    }
    CUDA_OK(cudaGetLastError());
    e->launches++;
  };
  // attention bias of the documents in `slots` (nullptr: all B)
  auto bias_build = [&](const int* slots, const int* n_act) {
    BiasArgs ba{};
    ba.bbox = bbox; ba.vis_bbox = e->vis_bbox.p; ba.t1 = e->bias_t1.p; ba.t2 = e->bias_t2.p;
    ba.lut1 = e->lut1.p; ba.lut2 = e->lut2.p; // every |rel| >= max_distance lands in the last bucket (HF:393-414), so the lookup index is clamped there: far keys
    // (most of them) then read the same table word, which the shared-memory crossbar broadcasts without a conflict
    ba.lut1_n = std::min(static_cast<int>(e->lut1.n), d.max_rel + 1);
    ba.lut2_n = std::min(static_cast<int>(e->lut2.n), d.max_rel2d + 1);
    ba.maskadd = e->maskadd.p;
    ba.bins1 = d.rel_bins; ba.bins2 = d.rel2d_bins; ba.heads = heads; ba.t2_pitch = bias_table_pitch(heads); ba.n_text = T; ba.seq = S; ba.pitch = e->bias_pitch;
    ba.kv_pitch = e->kv_pitch; ba.B = B; ba.out = e->BIAS.p; ba.slot_doc = slots; ba.n_active_dev = n_act;
    ba.doc_len = e->doc_len.p; ba.kept_idx = e->kept_idx.p; ba.n_vis = e->n_vis;
    const size_t smem = bias_build_smem(ba);
    static bool configured_dev[64] = {};
    bool& configured = configured_dev[e->device & 63];   // the attribute is per device
    if (!configured) {
      CUDA_OK(cudaFuncSetAttribute(bias_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      configured = true;
    }
    if (smem > 200 * 1024) throw std::runtime_error("relative-position tables do not fit shared memory");
    if (split) {
      const int work = S * (e->bias_pitch >> 3);
      bias_build_split_kernel<<<dim3((work + 255) / 256, B), 256, 0, st>>>(ba, e->bias_tx.p, e->bias_ty.p, e->BIASlo.p);
    } else {
      bias_build_kernel<<<e->sms, BIAS_THREADS, smem, st>>>(ba);
    }
    CUDA_OK(cudaGetLastError());
    e->launches++;
  };
  // vision branch for all B documents (EE/models/LayoutLMv3.py:358-373): patches -> conv GEMM (+bias, +pos_embed) ->
  // `norm`; X != nullptr: also the model LayerNorm into the fused rows
  auto vision = [&](RowOut xo, bool keep_normed) {
    const int per_doc = e->n_patch * e->kdim_patch / 4;
    if (e->px_async) CUDA_OK(cudaStreamWaitEvent(st, e->px_wait ? e->px_wait : e->px_ready, 0));
    im2col_kernel<<<dim3((per_doc + 255) / 256, B), 256, 0, st>>>(px, e->PATCH.p, split ? e->PATCHlo.p : nullptr, B,
                                                                 d.image, d.patch, d.channels);
    e->launches++;
    GemmArgs ga{};
    ga.m_dev = nullptr; ga.m_static = B * e->n_patch; ga.N = H; ga.K = e->kdim_patch; ga.bias = e->patch_b.p;
    ga.out = e->VIS.p; ga.ld_out = H; ga.pos = e->pos_embed.p; ga.n_patch = e->n_patch; ga.n_vis = e->n_vis;
    run_gemm<EPI_PATCH>(e, e->bn_h, e->t_patch, e->t_patch_w, e->t_patch_lo, e->t_patch_w_lo, ga, st);
    const int blocks = std::min((B * e->n_vis + 7) / 8, e->sms * 16);
    const int wp = keep_normed ? 1 : 0;
    switch (H % 128 == 0 ? H / 128 : 0) {
      case 1: visual_ln_vec_kernel<1><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 2: visual_ln_vec_kernel<2><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 3: visual_ln_vec_kernel<3><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 4: visual_ln_vec_kernel<4><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 5: visual_ln_vec_kernel<5><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 6: visual_ln_vec_kernel<6><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 7: visual_ln_vec_kernel<7><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      case 8: visual_ln_vec_kernel<8><<<blocks, 256, 0, st>>>(e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps); break;
      default:
        launch_nv(H, [&](auto nv) {
          visual_ln_kernel<decltype(nv)::value><<<(B * e->n_vis + 7) / 8, 256, 0, st>>>(
              e->VIS.p, ew, xo, wp, B, e->n_vis, T, S, H, d.vis_ln_eps, d.ln_eps);
        });
    }
    CUDA_OK(cudaGetLastError());
    e->launches++;
  };
  // X[slot, off .. off+rows) = LN_model(src rows of the survivors)  (H % 128 == 0 is checked at mmee_create)
  auto embed_finish = [&](const float* src, int rows, const int* map, int off, const int* n_act) {
    const int blocks = std::min((B * rows + 7) / 8, e->sms * 16);
    switch (H / 128) {
      case 1: embed_finish_vec_kernel<1><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 2: embed_finish_vec_kernel<2><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 3: embed_finish_vec_kernel<3><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 4: embed_finish_vec_kernel<4><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 5: embed_finish_vec_kernel<5><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 6: embed_finish_vec_kernel<6><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 7: embed_finish_vec_kernel<7><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      case 8: embed_finish_vec_kernel<8><<<blocks, 256, 0, st>>>(src, rows, map, ew, xout(cur), off, S, H, d.ln_eps, n_act); break;
      default: throw std::runtime_error("embedding-level exits need hidden % 128 == 0 and hidden <= 1024");
    }
    CUDA_OK(cudaGetLastError());
    e->launches++;
  };

  if (T > 0) {   // image-only engines (n_text = 0, BASELINE config 5) have no text tokens
    posid_kernel<<<(B + 7) / 8, 256, 0, st>>>(ids, e->posid.p, B, T, d.pad_id);
    e->launches++;
  }
  keymask_kernel<<<B, e->kv_pitch, 0, st>>>(mask, e->maskadd.p, e->kept_idx.p, e->doc_len.p, T, S, e->kv_pitch);
  e->launches++;

  const bool modality_exits = e->has_vision_exit || e->has_text_exit;
  bool any_embedding_exit = false;
  if (!modality_exits) {
    // pixel-independent work first: on the host path the pixel upload (96 % of the input bytes) overlaps it
    if (T > 0) text_embed(nullptr, nullptr, xout(0), nullptr);
    bias_build(nullptr, nullptr);
    vision(xout(0), false);
    mark(e, "embed", st);
    // text_visual_concat exit (EE/models/LayoutLMv3.py:581-606): mean over the 709 fused tokens after the model LayerNorm
    if (exit_no < E && d.exit_after_layer[exit_no] == 0) {
      meanpool_kernel<<<dim3((H + 31) / 32, B), 256, 0, st>>>(e->X[cur].p, split ? e->X32[cur].p : nullptr, e->POOL.p, S, H);
      e->launches++;
      run_exit(e->POOL.p, H, nullptr, nullptr, e->exit_heads[exit_no], false, nullptr);
      any_embedding_exit = true;
    }
  } else {
    // Embedding-level exits in the reference's order (EE/models/LayoutLMv3.py:441-606): vision branch -> vision_avg
    // exit -> text embeddings -> text_avg exit -> cat + model LayerNorm -> text_visual_concat exit.  In early-exit mode
    // every step after an exit runs on the survivors only: a document that leaves at vision_avg never gets text
    // embeddings, fused rows or an attention bias (true skipping, SURVEY.md §8 f3).
    vision(RowOut{nullptr, nullptr, nullptr}, true);                                   // VIS = norm(cls | patches + pos_embed), all documents
    if (exit_no < E && d.exit_after_layer[exit_no] == MMEE_EXIT_VISION_AVG) {
      meanpool_f32_kernel<<<dim3((H + 31) / 32, B), 256, 0, st>>>(e->VIS.p, e->POOLV.p, e->n_vis, H);   // :465-468, by document
      e->launches++;
      run_exit(e->POOLV.p, H, nullptr, nullptr, e->exit_heads[exit_no], false, e->slot_doc[sd].p);
    }
    // text embeddings of the survivors (before the model LayerNorm), indexed by their current slot
    const int* txt_map = nullptr;
    if (T > 0) text_embed(e->slot_doc[sd].p, e->n_dev.p + stage, RowOut{nullptr, nullptr, nullptr}, e->TXT.p);
    if (exit_no < E && d.exit_after_layer[exit_no] == MMEE_EXIT_TEXT_AVG) {
      meanpool_f32_kernel<<<dim3((H + 31) / 32, B), 256, 0, st>>>(e->TXT.p, e->POOLT.p, T, H);           // :519-521, by slot
      e->launches++;
      run_exit(e->POOLT.p, H, nullptr, nullptr, e->exit_heads[exit_no], false, nullptr);
      if (leave) txt_map = e->slot_src.p;                             // new slot -> slot the TXT rows were written under
    }
    // fused rows of the survivors: [text | visual] -> model LayerNorm (:549-566)
    if (T > 0) embed_finish(e->TXT.p, T, txt_map, 0, e->n_dev.p + stage);
    embed_finish(e->VIS.p, e->n_vis, e->slot_doc[sd].p, T, e->n_dev.p + stage);
    mark(e, "embed", st);
    if (exit_no < E && d.exit_after_layer[exit_no] == 0) {
      meanpool_kernel<<<dim3((H + 31) / 32, B), 256, 0, st>>>(e->X[cur].p, split ? e->X32[cur].p : nullptr, e->POOL.p, S, H);   // by slot
      e->launches++;
      run_exit(e->POOL.p, H, nullptr, nullptr, e->exit_heads[exit_no], false, nullptr);
      any_embedding_exit = true;
    }
  }
  // ---- dense embedding output -> ragged encoder input.  The embedding stage (and its mean-pool exits, which average
  // over ALL 709 tokens, pads included, as the reference does) works on dense [slot, 709] rows; from here on a document
  // owns only the rows of its kept tokens.  The same pass moves the survivors of the concat exit to their new slots.
  {
    launch_plan_rows(e->slot_doc[sd].p, e->doc_len.p, e->n_dev.p + stage, plan_view(e, rp), e->m_dev.p + stage, ATT_BQ, st);
    // where the dense rows of slot s live: by document (no vision / text exit: the embedding stage ran in document
    // order), else by the slot numbering of the embedding stage (identity, or new -> old after the concat exit left)
    const int* src_index = !modality_exits ? e->slot_doc[sd].p : ((any_embedding_exit && leave) ? e->slot_src.p : nullptr);
    auto gather = [&](const void* src, void* dst, int elem) {
      ragged_gather_kernel<<<dim3(16, B), 256, 0, st>>>(src, dst, src_index, e->slot_doc[sd].p, e->n_dev.p + stage,
                                                       e->plan_row0[rp].p, e->doc_len.p, e->kept_idx.p, T, e->n_vis, S, H * elem);
      e->launches++;
    };
    gather(e->X[cur].p, e->X[cur ^ 1].p, 2);
    if (split) {
      gather(e->Xlo[cur].p, e->Xlo[cur ^ 1].p, 2);
      gather(e->X32[cur].p, e->X32[cur ^ 1].p, 4);
    }
    CUDA_OK(cudaGetLastError());
    e->launches++;
    cur ^= 1;
  }
  if (modality_exits) {
    bias_build(e->slot_doc[sd].p, e->n_dev.p + stage);               // survivors only
    mark(e, "embed", st);                                             // (the embedding-level exits are part of this stage)
  } else if (any_embedding_exit) {
    mark(e, "exit", st);
  }

  // ---- encoder layers
  for (int l = 0; l < e->L; ++l) {
    LayerW& w = e->layers[l];
    const int* mdev = e->m_dev.p + stage;
    GemmArgs ga{};
    ga.m_dev = mdev; ga.N = 3 * H; ga.K = H; ga.bias = w.bqkv.p; ga.out = e->QK.p; ga.out_lo = e->QKlo.p; ga.ld_out = 2 * H;
    ga.vt = e->VT.p; ga.vt_lo = e->VTlo.p; ga.qk_cols = 2 * H; ga.row0 = e->plan_row0[rp].p; ga.n_slots_dev = e->n_dev.p + stage;
    ga.kv_pitch = e->kv_pitch; ga.heads = heads;
    run_gemm<EPI_QKV>(e, e->bn_qkv, e->t_x[cur], w.t_wqkv, e->t_x_lo[cur], w.t_wqkv_lo, ga, st);
    mark(e, "gemm", st);

    AttArgs aa;
    aa.slot_meta = e->plan_meta[rp].p; aa.qt_slot = e->plan_qt_slot[rp].p; aa.n_qt_dev = e->plan_n_qt[rp].p;
    aa.ctx = e->CTX.p; aa.ctx_lo = e->CTXlo.p; aa.H = H; aa.heads = heads; aa.seq = S;
    aa.tail16 = (e->tail16 && !split) ? 1 : 0;
    aa.experiment = getenv("MMEE_ATT_EXPERIMENT") ? atoi(getenv("MMEE_ATT_EXPERIMENT")) : 0; aa.err_flag = e->err_flags.p; aa.trace = e->att_trace.p;
    // developer experiment MMEE_ATT_ONE_CTA=1: one attention CTA per SM (extra dynamic shared memory keeps the second
    // one out) — shows what a softmax warp does when it has its scheduler's MUFU to itself
    static const bool one_cta = getenv("MMEE_ATT_ONE_CTA") != nullptr;
    launch_attention(e->device, e->sms, e->att_maps, aa, split, e->trace_on && l == 0, one_cta, st);
    e->launches++;
    mark(e, "attention", st);

    // y_resid: the out-projection writes Y2 (Y still holds the previous layer's MLP-down sums, from which this residual
    // is recomputed through the row map the last LayerNorm left); the first layer adds the embedding output itself
    const bool yr = e->y_resid;
    // developer A/B switch, off: prefetching the next tile's residual rows into L2 made the GEMM stage 0.4 ms slower
    static const int resid_pf = getenv("MMEE_RESID_PREFETCH") ? atoi(getenv("MMEE_RESID_PREFETCH")) : 0;
    float* y_att = yr ? e->Y2.p : e->Y.p;
    ga = GemmArgs{};
    ga.m_dev = mdev; ga.N = H; ga.K = H; ga.bias = w.bo.p; ga.out = y_att; ga.ld_out = H; ga.resid = e->X[cur].p;
    ga.resid_lo = (x_lo_valid && !yr) ? e->Xlo[cur].p : nullptr;
    ga.resid_f32 = split ? e->X32[cur].p : nullptr;
    if (yr && x_lo_valid) {
      const LayerW& pw = e->layers[l - 1];
      ga.resid = nullptr; ga.resid_prefetch = resid_pf;
      ga.resid_y = e->Y.p; ga.resid_stats = e->ln_stats2.p; ga.resid_src = e->ln_src2.p;
      ga.resid_w = pw.ln2_w.p; ga.resid_b = pw.ln2_b.p;
    }
    run_gemm<EPI_RESID_F32>(e, e->bn_h, e->t_ctx, w.t_wo, e->t_ctx_lo, w.t_wo_lo, ga, st);
    mark(e, "gemm", st);
    launch_ln(e, y_att, e->A1.p, yr ? nullptr : e->A1lo.p, split ? e->A132.p : nullptr, w.ln1_w.p, w.ln1_b.p, B, mdev, nullptr,
              plan_view(e, rp), plan_view(e, rp), e->n_dev.p + stage, st, yr ? e->ln_stats1.p : nullptr, nullptr);
    e->launches++;
    mark(e, "norm", st);

    ga = GemmArgs{};
    ga.m_dev = mdev; ga.N = I; ga.K = H; ga.bias = w.bi.p; ga.out = e->MID.p; ga.out_lo = e->MIDlo.p; ga.ld_out = I;
    run_gemm<EPI_GELU_BF16>(e, e->bn_i, e->t_a1, w.t_wi, e->t_a1_lo, w.t_wi_lo, ga, st);
    ga = GemmArgs{};
    ga.m_dev = mdev; ga.N = H; ga.K = I; ga.bias = w.bo2.p; ga.out = e->Y.p; ga.ld_out = H; ga.resid = e->A1.p;
    ga.resid_lo = yr ? nullptr : e->A1lo.p;
    ga.resid_f32 = split ? e->A132.p : nullptr;
    if (yr) {                                     // residual = LayerNorm1(Y2), same rows
      ga.resid = nullptr; ga.resid_prefetch = resid_pf;
      ga.resid_y = e->Y2.p; ga.resid_stats = e->ln_stats1.p; ga.resid_src = nullptr;
      ga.resid_w = w.ln1_w.p; ga.resid_b = w.ln1_b.p;
    }
    if (split && e->n_kchunks > 1) {
      // K chunks: Y = A1 + b + MID[:, 0:kc] W[:, 0:kc]^T, then Y += MID[:, c] W[:, c]^T in fp32 (see kchunk)
      for (int c = 0; c < e->n_kchunks; ++c) {
        ga.K = e->kchunk;
        if (c > 0) { ga.bias = e->zero_bias.p; ga.resid_f32 = e->Y.p; }
        run_gemm<EPI_RESID_F32>(e, e->bn_h, e->t_mid_c[c], w.t_wo2_c[c], e->t_mid_lo_c[c], w.t_wo2_lo_c[c], ga, st);
      }
    } else {
      run_gemm<EPI_RESID_F32>(e, e->bn_h, e->t_mid, w.t_wo2, e->t_mid_lo, w.t_wo2_lo, ga, st);
    }
    mark(e, "gemm", st);

    const bool last = (l == e->L - 1);
    const bool exit_here = (exit_no < E && d.exit_after_layer[exit_no] == l + 1);
    const int* ln_src = nullptr;
    const int y_rp = rp;                          // row plan under which Y was written
    if (exit_here) {
      run_exit(e->Y.p, 0, w.ln2_w.p, w.ln2_b.p, e->exit_heads[exit_no], false, nullptr, e->plan_row0[y_rp].p);
      if (leave) ln_src = e->slot_src.p;
      mark(e, "exit", st);
    }
    if (!last) {
      launch_ln(e, e->Y.p, e->X[cur ^ 1].p, yr ? nullptr : e->Xlo[cur ^ 1].p, split ? e->X32[cur ^ 1].p : nullptr, w.ln2_w.p,
                w.ln2_b.p, B, e->m_dev.p + stage, ln_src, plan_view(e, rp), plan_view(e, y_rp), e->n_dev.p + stage, st,
                yr ? e->ln_stats2.p : nullptr, yr ? e->ln_src2.p : nullptr);
      e->launches++;
      cur ^= 1;
      x_lo_valid = e->precise_residual;
      mark(e, "norm", st);
    } else {
      // final classifier on the CLS row of the last layer (EE/models/LayoutLMv3.py:730-731); rows still live in
      // Y under the row plan of before the compaction when an exit was just taken at layer L.
      run_exit(e->Y.p, 0, w.ln2_w.p, w.ln2_b.p, e->classifier, true, ln_src, e->plan_row0[y_rp].p);
      mark(e, "exit", st);
    }
  }

  // ---- results (device -> caller's device buffers)
  if (cap && st != cap->root) {            // close the innermost IF body: the rest follows the outermost IF node
    cudaGraph_t done = nullptr;
    CUDA_OK(cudaStreamEndCapture(st, &done));
    st = cap->root;
  }
  hist_to_i64_kernel<<<1, 64, 0, st>>>(e->hist.p, e->hist64.p, E1);
  e->launches++;
  auto d2d = [&](void* dst, const void* src, size_t bytes) {     // the host path hands in the engine's own buffers
    if (dst && dst != src) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st));
  };
  d2d(out->logits, e->out_logits.p, static_cast<size_t>(B) * K * 4);
  d2d(out->exit_index, e->out_exit.p, static_cast<size_t>(B) * 4);
  d2d(out->criterion, e->out_crit.p, static_cast<size_t>(B) * 4);
  d2d(out->all_exit_logits, e->all_logits.p, static_cast<size_t>(E1) * B * K * 4);
  d2d(out->all_head_logits, e->all_head.p, static_cast<size_t>(E1) * B * K * 4);
  d2d(out->all_criteria, e->all_crit.p, static_cast<size_t>(E1) * B * 4);
  d2d(out->exit_hist, e->hist64.p, static_cast<size_t>(E1) * 8);
  mark(e, "end", st);
  if (!cap) CUDA_OK(cudaEventRecord(e->last_done, st));
}

// Device-side error flags, turned into errors by the synchronous entry points instead of returning garbage:
// [0] guard of the attention kernel's online softmax (a deferred rescale factor underflowed; unreachable by
// construction, see ATT_JUMP in attention.cuh); [1] an input_id / bbox coordinate outside its embedding table (the
// reference raises IndexError there; the kernels clamp, so no out-of-bounds read happens).
void check_error_flags(mmee_engine* e) {
  int flags[2] = {0, 0};
  CUDA_OK(cudaMemcpy(flags, e->err_flags.p, sizeof(flags), cudaMemcpyDeviceToHost));
  if (flags[0] || flags[1]) {
    CUDA_OK(cudaMemset(e->err_flags.p, 0, sizeof(flags)));
    if (flags[1])
      throw std::runtime_error("input out of range: input_ids must lie in [0, vocab) and bbox coordinates in [0, max_2d)");
    throw std::runtime_error("attention online-softmax guard tripped (rescale factor underflow)");
  }
}

// Folds the stage events of every forward recorded since the last call into per-stage SUMS (ms) plus the number of
// forwards ("forwards"); callers divide.  The interval between one forward's "end" and the next one's "start" is not
// a stage.  No new events -> the previous result stays.
void collect_profile(mmee_engine* e) {
  if (!e->profiling || e->ev.size() < 2) return;
  e->stage_ms.clear();
  double total = 0, forwards = 0;
  for (size_t i = 0; i < e->ev.size(); ++i) {
    if (e->ev[i].first == "start") { forwards += 1; continue; }
    if (i == 0) continue;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e->ev[i - 1].second, e->ev[i].second) != cudaSuccess) continue;
    e->stage_ms[e->ev[i].first] += ms;
    total += ms;
  }
  e->stage_ms["total"] = total;
  e->stage_ms["forwards"] = forwards;
  for (auto& x : e->ev) cudaEventDestroy(x.second);
  e->ev.clear();
}

// staged inputs of the host paths and of plans, for max_batch documents
void alloc_inputs(mmee_engine* e) {
  if (e->in_ids.p) return;
  const size_t mb = e->max_batch, T = e->T;
  e->in_ids.alloc(mb * T); e->in_bbox.alloc(mb * T * 4); e->in_mask.alloc(mb * T);
  e->in_px.alloc(mb * e->d.channels * e->d.image * e->d.image);
}

// uint8 images (mmee_images, image.cuh): every check runs on the host, before anything is enqueued
void check_images(const mmee_engine* e, int B, const mmee_images* im) {
  if (!im || !im->data || !im->offsets || !im->sizes) throw std::runtime_error("images: data, offsets and sizes are required");
  if (e->d.channels != 3)
    throw std::runtime_error("uint8 images need an engine with channels = 3, this one has " + std::to_string(e->d.channels));
  if (B < 1 || B > e->max_batch) throw std::runtime_error("batch out of range");
  if (im->channels != 1 && im->channels != 3)
    throw std::runtime_error("images: channels must be 1 (grayscale) or 3 (RGB), got " + std::to_string(im->channels));
  for (int b = 0; b < B; ++b) {
    const int h = im->sizes[2 * b], w = im->sizes[2 * b + 1];
    if (h < 1 || h > IMG_MAX_SIDE || w < 1 || w > IMG_MAX_SIDE)
      throw std::runtime_error("image " + std::to_string(b) + ": size (" + std::to_string(h) + ", " + std::to_string(w) +
                               ") outside [1, " + std::to_string(IMG_MAX_SIDE) + "]");
    const int64_t off = im->offsets[b], n = static_cast<int64_t>(h) * w * im->channels;
    if (off < 0 || off > im->total_bytes - n)
      throw std::runtime_error("image " + std::to_string(b) + ": bytes [" + std::to_string(off) + ", " +
                               std::to_string(off + n) + ") run past total_bytes = " + std::to_string(im->total_bytes));
  }
}

// Enqueues the preprocess of a checked batch on `st`: packed bytes `data` (device) -> px f32 [B, 3, S, S] (device).
// Coefficient tables are computed once per distinct input length; scratch grows, it is never allocated per call.
void preprocess_images(mmee_engine* e, int B, const mmee_images* im, const uint8_t* data, float* px, cudaStream_t st) {
  const int S = e->d.image, C = im->channels;
  const size_t desc_bytes = sizeof(ImageDesc) * e->max_batch, meta_bytes = desc_bytes + sizeof(ImageAxis) * 2 * e->max_batch;
  if (!e->img_meta_host) {
    CUDA_OK(cudaMallocHost(&e->img_meta_host, meta_bytes));
    e->img_meta.alloc(meta_bytes);
    e->img_bounds.alloc(static_cast<size_t>(2) * e->max_batch * S);
    CUDA_OK(cudaEventCreateWithFlags(&e->img_meta_copied, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&e->img_done, cudaEventDisableTiming));
  }
  std::vector<ImageDesc> desc(B);
  std::vector<ImageAxis> axes;
  std::map<int, int> table;                 // input length -> coefficient table
  int64_t kk_n = 0, tmp_n = 0, max_items = 0;
  auto axis = [&](int in) {
    auto it = table.find(in);
    if (it != table.end()) return it->second;
    const int ksize = 2 * std::max(1, (in + S - 1) / S) + 1;   // Pillow: 2 ceil(max(in / S, 1)) + 1
    axes.push_back(ImageAxis{in, ksize, kk_n});
    kk_n += static_cast<int64_t>(S) * ksize;
    return table[in] = static_cast<int>(axes.size()) - 1;
  };
  for (int b = 0; b < B; ++b) {
    ImageDesc& dsc = desc[b];
    dsc.h = im->sizes[2 * b]; dsc.w = im->sizes[2 * b + 1];
    dsc.src_off = im->offsets[b];
    dsc.th = axis(dsc.h); dsc.tw = axis(dsc.w);
    // Pillow's Image.resize shrinks a page more than 100 times taller than wide vertically first
    dsc.vfirst = dsc.h > 100 * dsc.w && S < dsc.h;
    dsc.pad_ = 0;
    const int64_t items = dsc.vfirst ? static_cast<int64_t>(S) * dsc.w : static_cast<int64_t>(dsc.h) * S;
    dsc.tmp_off = tmp_n;
    tmp_n += items * C;
    max_items = std::max(max_items, items);
  }
  if (static_cast<int64_t>(e->img_kk.n) < kk_n || static_cast<int64_t>(e->img_tmp.n) < tmp_n) {
    CUDA_OK(cudaEventSynchronize(e->img_done));             // a preprocess on another stream may still read them
    if (static_cast<int64_t>(e->img_kk.n) < kk_n) e->img_kk.alloc(kk_n);
    if (static_cast<int64_t>(e->img_tmp.n) < tmp_n) e->img_tmp.alloc(tmp_n);
  }
  CUDA_OK(cudaEventSynchronize(e->img_meta_copied));        // the staging buffer is free again
  memcpy(e->img_meta_host, desc.data(), sizeof(ImageDesc) * B);
  memcpy(e->img_meta_host + desc_bytes, axes.data(), sizeof(ImageAxis) * axes.size());
  CUDA_OK(cudaStreamWaitEvent(st, e->img_done, 0));
  CUDA_OK(cudaMemcpyAsync(e->img_meta.p, e->img_meta_host, meta_bytes, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaEventRecord(e->img_meta_copied, st));
  const auto* d_desc = reinterpret_cast<const ImageDesc*>(e->img_meta.p);
  const auto* d_axes = reinterpret_cast<const ImageAxis*>(e->img_meta.p + desc_bytes);
  image_coeffs_kernel<<<static_cast<unsigned>(axes.size()), 128, 0, st>>>(d_axes, S, e->img_bounds.p, e->img_kk.p);
  const unsigned gy = static_cast<unsigned>(std::min(B, 65535));
  const dim3 g1(static_cast<unsigned>(std::min<int64_t>((max_items + 255) / 256, 1024)), gy);
  const dim3 g2(static_cast<unsigned>(std::min<int64_t>((static_cast<int64_t>(S) * S + 255) / 256, 1024)), gy);
  if (C == 1) {
    image_pass1_kernel<1><<<g1, 256, 0, st>>>(data, d_desc, B, S, d_axes, e->img_bounds.p, e->img_kk.p, e->img_tmp.p);
    image_pass2_kernel<1><<<g2, 256, 0, st>>>(e->img_tmp.p, d_desc, B, S, d_axes, e->img_bounds.p, e->img_kk.p, px);
  } else {
    image_pass1_kernel<3><<<g1, 256, 0, st>>>(data, d_desc, B, S, d_axes, e->img_bounds.p, e->img_kk.p, e->img_tmp.p);
    image_pass2_kernel<3><<<g2, 256, 0, st>>>(e->img_tmp.p, d_desc, B, S, d_axes, e->img_bounds.p, e->img_kk.p, px);
  }
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaEventRecord(e->img_done, st));
}

// mmee_forward / mmee_forward_images: inputs and outputs in host memory.  The small inputs go up on the engine's
// stream; `stage_pixels(copy_stream)` enqueues what fills in_px (96 % of the bytes), which overlaps the text embedding
// and bias build and is first needed by im2col.
template <typename F>
void host_forward(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                  const mmee_policy* policy, const mmee_outputs* out, F&& stage_pixels) {
  const int T = e->T, K = e->K, E1 = e->d.n_exits + 1;
  const size_t n_ids = static_cast<size_t>(B) * T;
  alloc_inputs(e);
  cudaStream_t st = e->stream;
  // a plan run on another stream may still read the staged inputs
  CUDA_OK(cudaStreamWaitEvent(st, e->last_done, 0));
  // small inputs first (one H2D copy engine serves both streams in issue order)
  CUDA_OK(cudaMemcpyAsync(e->in_ids.p, input_ids, n_ids * 8, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->in_bbox.p, bbox, n_ids * 32, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemcpyAsync(e->in_mask.p, attention_mask, n_ids * 8, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaEventRecord(e->fwd_start, st));
  CUDA_OK(cudaStreamWaitEvent(e->copy_stream, e->fwd_start, 0));       // previous forward has released in_px
  stage_pixels(e->copy_stream);
  CUDA_OK(cudaEventRecord(e->px_ready, e->copy_stream));
  e->px_async = true;
  // run with outputs in the engine's own device buffers, then copy what was asked for to the host
  mmee_outputs dv{};
  dv.logits = e->out_logits.p; dv.exit_index = e->out_exit.p; dv.criterion = e->out_crit.p;
  dv.exit_hist = reinterpret_cast<int64_t*>(e->hist64.p);
  if (out->all_exit_logits) dv.all_exit_logits = e->all_logits.p;
  if (out->all_head_logits) dv.all_head_logits = e->all_head.p;
  if (out->all_criteria) dv.all_criteria = e->all_crit.p;
  try {
    forward_device(e, B, e->in_ids.p, e->in_bbox.p, e->in_mask.p, e->in_px.p, policy, &dv, st);
  } catch (...) {
    e->px_async = false;
    throw;
  }
  e->px_async = false;
  CUDA_OK(cudaMemcpyAsync(out->logits, dv.logits, static_cast<size_t>(B) * K * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaMemcpyAsync(out->exit_index, dv.exit_index, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, st));
  if (out->criterion) CUDA_OK(cudaMemcpyAsync(out->criterion, dv.criterion, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost, st));
  if (out->exit_hist) CUDA_OK(cudaMemcpyAsync(out->exit_hist, dv.exit_hist, static_cast<size_t>(E1) * 8, cudaMemcpyDeviceToHost, st));
  if (out->all_exit_logits) CUDA_OK(cudaMemcpyAsync(out->all_exit_logits, dv.all_exit_logits, static_cast<size_t>(E1) * B * K * 4, cudaMemcpyDeviceToHost, st));
  if (out->all_head_logits) CUDA_OK(cudaMemcpyAsync(out->all_head_logits, dv.all_head_logits, static_cast<size_t>(E1) * B * K * 4, cudaMemcpyDeviceToHost, st));
  if (out->all_criteria) CUDA_OK(cudaMemcpyAsync(out->all_criteria, dv.all_criteria, static_cast<size_t>(E1) * B * 4, cudaMemcpyDeviceToHost, st));
  CUDA_OK(cudaStreamSynchronize(st));
  collect_profile(e);
  check_error_flags(e);
}

}  // namespace

// A captured and instantiated forward for one (B, criterion, mode, want_all): include/mmee.h mmee_plan_create.
struct mmee_plan {
  mmee_engine* e = nullptr;
  int B = 0, criterion = 0, mode = 0;
  bool want_all = false;
  DevBuf<float> policy_dev;                 // [2 (E+1)] {threshold, 1/T} per exit (exit_policy), read by the graph
  float* policy_host = nullptr;             // pinned staging of policy_dev
  cudaEvent_t policy_copied = nullptr;      // the previous run's upload of policy_host has completed
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  ~mmee_plan() {
    if (exec) cudaGraphExecDestroy(exec);
    if (graph) cudaGraphDestroy(graph);
    if (policy_copied) cudaEventDestroy(policy_copied);
    if (policy_host) cudaFreeHost(policy_host);
  }
};

namespace {

// One eager forward of B neutral documents (ids 0, boxes 0, mask 1, pixels 0): sets the kernel attributes (the
// first-launch blocks of the launch helpers) and loads every module, neither of which may happen during a capture.
void warm_up(mmee_engine* e, int B, int criterion) {
  const size_t n_ids = static_cast<size_t>(B) * e->T, n_px = static_cast<size_t>(B) * e->d.channels * e->d.image * e->d.image;
  cudaStream_t st = e->stream;
  CUDA_OK(cudaStreamWaitEvent(st, e->last_done, 0));
  std::vector<int64_t> ones(n_ids, 1);
  CUDA_OK(cudaMemsetAsync(e->in_ids.p, 0, n_ids * 8, st));
  CUDA_OK(cudaMemsetAsync(e->in_bbox.p, 0, n_ids * 32, st));
  CUDA_OK(cudaMemcpyAsync(e->in_mask.p, ones.data(), n_ids * 8, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaMemsetAsync(e->in_px.p, 0, n_px * 4, st));
  std::vector<float> thr(std::max(e->d.n_exits, 1), 0.f);
  const mmee_policy pol{criterion, 0, thr.data(), nullptr};
  mmee_outputs dv{};                        // with the all_* outputs: every kernel a plan can contain is launched
  dv.logits = e->out_logits.p; dv.exit_index = e->out_exit.p;
  dv.all_exit_logits = e->all_logits.p; dv.all_head_logits = e->all_head.p; dv.all_criteria = e->all_crit.p;
  forward_device(e, B, e->in_ids.p, e->in_bbox.p, e->in_mask.p, e->in_px.p, &pol, &dv, st);
  CUDA_OK(cudaStreamSynchronize(st));
  check_error_flags(e);
}

// Records forward_device for the plan into p->graph.  On failure every capture that was begun is ended and its graph
// dropped, so the streams and the engine stay usable.
void capture_plan(mmee_plan* p) {
  mmee_engine* e = p->e;
  Capture cap;
  cap.policy_dev = p->policy_dev.p;
  cap.skip_tail = p->mode == 1;
  std::vector<float> thr(std::max(e->d.n_exits, 1), 0.f);   // ignored: the graph reads policy_dev
  const mmee_policy pol{p->criterion, p->mode, thr.data(), nullptr};
  mmee_outputs dv{};                        // results stay in the engine's own buffers
  dv.logits = e->out_logits.p; dv.exit_index = e->out_exit.p; dv.criterion = e->out_crit.p;
  dv.exit_hist = reinterpret_cast<int64_t*>(e->hist64.p);
  if (p->want_all) { dv.all_exit_logits = e->all_logits.p; dv.all_head_logits = e->all_head.p; dv.all_criteria = e->all_crit.p; }
  // ends a capture left open by a failure (a body graph belongs to its IF node, the root graph to nobody) and frees the
  // stream
  auto drop = [](cudaStream_t s, bool root) {
    if (!s) return;
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &status) == cudaSuccess && status != cudaStreamCaptureStatusNone) {
      cudaGraph_t g = nullptr;
      cudaStreamEndCapture(s, &g);
      if (g && root) cudaGraphDestroy(g);
    }
    cudaStreamDestroy(s);
  };
  try {
    CUDA_OK(cudaStreamCreateWithFlags(&cap.root, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamCreateWithFlags(&cap.side[0], cudaStreamNonBlocking));
    CUDA_OK(cudaStreamCreateWithFlags(&cap.side[1], cudaStreamNonBlocking));
    CUDA_OK(cudaStreamBeginCapture(cap.root, cudaStreamCaptureModeThreadLocal));
    e->capturing = true;
    forward_device(e, p->B, e->in_ids.p, e->in_bbox.p, e->in_mask.p, e->in_px.p, &pol, &dv, cap.root, &cap);
    e->capturing = false;
    CUDA_OK(cudaStreamEndCapture(cap.root, &p->graph));
  } catch (...) {
    e->capturing = false;
    drop(cap.side[0], false); drop(cap.side[1], false); drop(cap.root, true);
    cudaGetLastError();
    throw;
  }
  drop(cap.side[0], false); drop(cap.side[1], false); drop(cap.root, true);
}

// One run of a plan on `st`: inputs into the engine's staging buffers, the policy into policy_dev, the graph, results
// out to the caller.  Ordered after the previous forward of the engine like every forward (last_done).
void plan_run(mmee_plan* p, const int64_t* ids, const int64_t* bbox, const int64_t* mask, const float* px,
              const mmee_policy* pol, const mmee_outputs* out, cudaStream_t st, bool host) {
  mmee_engine* e = p->e;
  const mmee_model_desc& d = e->d;
  const int B = p->B, T = e->T, K = e->K, E = d.n_exits, E1 = E + 1;
  if (!pol || (E > 0 && !pol->thresholds)) throw std::runtime_error("policy/thresholds missing");
  if (pol->criterion != p->criterion || pol->mode != p->mode)
    throw std::runtime_error("policy criterion / mode differ from the plan's (captured with criterion " +
                             std::to_string(p->criterion) + ", mode " + std::to_string(p->mode) + ")");
  if (!out || !out->logits || !out->exit_index) throw std::runtime_error("outputs missing");
  if (!p->want_all && (out->all_exit_logits || out->all_head_logits || out->all_criteria))
    throw std::runtime_error("all_* outputs need a plan created with want_all = 1");
  if (!ids && T > 0) throw std::runtime_error("inputs missing");
  if (!bbox && T > 0) throw std::runtime_error("inputs missing");
  if (!mask && T > 0) throw std::runtime_error("inputs missing");
  if (!px) throw std::runtime_error("inputs missing");
  const size_t n_ids = static_cast<size_t>(B) * T, n_px = static_cast<size_t>(B) * d.channels * d.image * d.image;
  const cudaMemcpyKind in_kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const cudaMemcpyKind out_kind = host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
  CUDA_OK(cudaEventSynchronize(p->policy_copied));           // the staging buffer is free again
  for (int x = 0; x < E1; ++x) exit_policy(e, pol, x, &p->policy_host[2 * x], &p->policy_host[2 * x + 1]);
  CUDA_OK(cudaStreamWaitEvent(st, e->last_done, 0));
  if (n_ids) {
    CUDA_OK(cudaMemcpyAsync(e->in_ids.p, ids, n_ids * 8, in_kind, st));
    CUDA_OK(cudaMemcpyAsync(e->in_bbox.p, bbox, n_ids * 32, in_kind, st));
    CUDA_OK(cudaMemcpyAsync(e->in_mask.p, mask, n_ids * 8, in_kind, st));
  }
  CUDA_OK(cudaMemcpyAsync(e->in_px.p, px, n_px * 4, in_kind, st));
  CUDA_OK(cudaMemcpyAsync(p->policy_dev.p, p->policy_host, static_cast<size_t>(E1) * 2 * 4, cudaMemcpyHostToDevice, st));
  CUDA_OK(cudaEventRecord(p->policy_copied, st));
  CUDA_OK(cudaGraphLaunch(p->exec, st));
  auto copy_out = [&](void* dst, const void* src, size_t bytes) {
    if (dst) CUDA_OK(cudaMemcpyAsync(dst, src, bytes, out_kind, st));
  };
  copy_out(out->logits, e->out_logits.p, static_cast<size_t>(B) * K * 4);
  copy_out(out->exit_index, e->out_exit.p, static_cast<size_t>(B) * 4);
  copy_out(out->criterion, e->out_crit.p, static_cast<size_t>(B) * 4);
  copy_out(out->all_exit_logits, e->all_logits.p, static_cast<size_t>(E1) * B * K * 4);
  copy_out(out->all_head_logits, e->all_head.p, static_cast<size_t>(E1) * B * K * 4);
  copy_out(out->all_criteria, e->all_crit.p, static_cast<size_t>(E1) * B * 4);
  copy_out(out->exit_hist, e->hist64.p, static_cast<size_t>(E1) * 8);
  CUDA_OK(cudaEventRecord(e->last_done, st));
}

void plan_destroy(mmee_plan* p) {
  mmee_engine* e = p->e;
  cudaSetDevice(e->device);
  cudaEventSynchronize(e->last_done);       // the graph may still be running on a caller's stream
  e->plans.erase(std::remove(e->plans.begin(), e->plans.end(), p), e->plans.end());
  delete p;
}

}  // namespace

// ================================================================================================ C ABI
#define MMEE_TRY try {
#define MMEE_CATCH                                  \
  }                                                 \
  catch (const std::exception& ex) {                \
    g_err = ex.what();                              \
    return -1;                                      \
  }                                                 \
  catch (...) {                                     \
    g_err = "unknown error";                        \
    return -2;                                      \
  }

extern "C" {

const char* mmee_last_error(void) { return g_err.c_str(); }
const char* mmee_version(void) { return "mmee-b200 0.1 (sm_100a)"; }

int mmee_create(const mmee_model_desc* desc, int device, int max_batch, mmee_engine** out) {
  MMEE_TRY
  if (!desc || !out) throw std::runtime_error("null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    throw std::runtime_error("no CUDA device: libmmee has no CPU fallback");
  CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_OK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) throw std::runtime_error(std::string("libmmee is built for sm_100a only; device is ") + prop.name);
  const mmee_model_desc& d = *desc;
  if (d.hidden % d.heads || d.hidden / d.heads != 64) throw std::runtime_error("head_dim must be 64");
  if (4 * d.coord + 2 * d.shape != d.hidden) throw std::runtime_error("4*coord + 2*shape != hidden");
  if (d.hidden % 128 || d.inter % 128 || d.hidden > 1024) throw std::runtime_error("hidden/inter must be multiples of 128, hidden <= 1024");
  if (d.n_labels > 32 || d.n_labels < 2) throw std::runtime_error("n_labels must be in [2, 32]");
  if (d.n_exits < 0 || d.n_exits > MMEE_MAX_EXITS) throw std::runtime_error("bad n_exits");
  for (int i = 0; i < d.n_exits; ++i) {
    if (d.exit_after_layer[i] < MMEE_EXIT_VISION_AVG || d.exit_after_layer[i] > d.layers) throw std::runtime_error("exit layer out of range");
    if (i && d.exit_after_layer[i] <= d.exit_after_layer[i - 1]) throw std::runtime_error("exits must be ascending");
  }
  if ((d.channels * d.patch * d.patch) % 64) throw std::runtime_error("patch K dim must be a multiple of 64");
  if (max_batch < 1) throw std::runtime_error("max_batch < 1");
  auto* e = new mmee_engine();
  e->d = d;
  e->device = device;
  e->max_batch = max_batch;
  if (d.compute_dtype != MMEE_DTYPE_BF16 && d.compute_dtype != MMEE_DTYPE_FP32) throw std::runtime_error("compute_dtype must be MMEE_DTYPE_BF16 or MMEE_DTYPE_FP32");
  if (d.n_text > 0 && d.n_text + d.pad_id + 1 > d.max_pos) throw std::runtime_error("n_text + pad_id + 1 exceeds max_pos (position table too small)");
  e->split = d.compute_dtype == MMEE_DTYPE_FP32;
  e->H = d.hidden; e->L = d.layers; e->heads = d.heads; e->I = d.inter; e->T = d.n_text; e->K = d.n_labels;
  e->n_patch = (d.image / d.patch) * (d.image / d.patch);
  e->n_vis = e->n_patch + 1;
  e->S = e->T + e->n_vis;
  e->kdim_patch = d.channels * d.patch * d.patch;
  e->kv_pitch = ((e->S + 127) / 128) * 128;
  e->bias_pitch = ((e->S + ATT_BKV - 1) / ATT_BKV) * ATT_BKV;   // whole key tiles: the pitch padding carries the -60000 mask
  // a last key tile with <= 16 real keys (an unpadded document, S = 709: 5) runs as a 16-key tile (N = 16 MMAs, a quarter of
  // the softmax work); decided per document by the attention kernel (documents are ragged)
  e->tail16 = !getenv("MMEE_NO_TAIL16");
  if (e->kv_pitch > 1024) throw std::runtime_error("sequence too long for keymask_kernel");
  e->sms = prop.multiProcessorCount;
  if (const char* pr = getenv("MMEE_PRECISE_RESIDUAL")) e->precise_residual = pr[0] != '0';   // developer A/B switch
  if (e->split) e->precise_residual = true;   // fp32 engine mode: split operands everywhere (and full 64-key tiles in attention)
  e->y_resid = e->precise_residual && !e->split && e->H % 128 == 0;
  if (const char* yr = getenv("MMEE_Y_RESID")) e->y_resid = e->y_resid && yr[0] != '0';   // developer A/B switch
  e->bn_h = gemm_block_n(e->H); e->bn_qkv = gemm_block_n_qkv(e->H); e->bn_i = gemm_block_n(e->I);
  try {
    CUDA_OK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUDA_OK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    CUDA_OK(cudaEventCreateWithFlags(&e->px_ready, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&e->fwd_start, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&e->last_done, cudaEventDisableTiming));
    allocate(e);
  } catch (...) {
    delete e;
    throw;
  }
  *out = e;
  return 0;
  MMEE_CATCH
}

void mmee_destroy(mmee_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  while (!e->plans.empty()) plan_destroy(e->plans.back());
  delete e;
}

int mmee_set_weight(mmee_engine* e, const char* hf_name, const float* host_data, const int64_t* shape, int rank) {
  MMEE_TRY
  if (!e || !hf_name || !host_data) throw std::runtime_error("null argument");
  size_t n = 1;
  std::vector<int64_t> sh;
  for (int i = 0; i < rank; ++i) { n *= static_cast<size_t>(shape[i]); sh.push_back(shape[i]); }
  e->raw[hf_name].assign(host_data, host_data + n);
  e->raw_shape[hf_name] = sh;
  e->finalized = false;
  return 0;
  MMEE_CATCH
}

int mmee_set_bucket_lut(mmee_engine* e, int which, const uint8_t* lut, int n) {
  MMEE_TRY
  if (!e || !lut || n < 1) throw std::runtime_error("bad argument");
  (which == 0 ? e->h_lut1 : e->h_lut2).assign(lut, lut + n);
  e->finalized = false;
  return 0;
  MMEE_CATCH
}

int mmee_get_bucket_lut(mmee_engine* e, int which, uint8_t* lut_out, int capacity) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  std::vector<uint8_t> t = which == 0 ? e->h_lut1 : e->h_lut2;
  if (t.empty()) t = which == 0 ? default_lut(e->d.rel_bins, e->d.max_rel, 1024) : default_lut(e->d.rel2d_bins, e->d.max_rel2d, 1024);
  const int n = static_cast<int>(t.size());
  if (lut_out) memcpy(lut_out, t.data(), std::min(n, capacity));
  return n;
  MMEE_CATCH
}

int mmee_finalize_weights(mmee_engine* e) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  finalize(e);
  return 0;
  MMEE_CATCH
}

int mmee_forward_device(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                        const int64_t* attention_mask, const float* pixel_values, const mmee_policy* policy,
                        const mmee_outputs* out, void* cuda_stream) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  CUDA_OK(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : e->stream;
  forward_device(e, B, input_ids, bbox, attention_mask, pixel_values, policy, out, st);
  if (!cuda_stream) {
    CUDA_OK(cudaStreamSynchronize(st));
    collect_profile(e);
    check_error_flags(e);
  }
  return 0;
  MMEE_CATCH
}

int mmee_forward(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                 const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out) {
  MMEE_TRY
  if (!e || !out) throw std::runtime_error("null argument");
  if (B < 1 || B > e->max_batch) throw std::runtime_error("batch out of range");
  CUDA_OK(cudaSetDevice(e->device));
  const size_t n_px = static_cast<size_t>(B) * e->d.channels * e->d.image * e->d.image;
  host_forward(e, B, input_ids, bbox, attention_mask, policy, out, [&](cudaStream_t cs) {
    CUDA_OK(cudaMemcpyAsync(e->in_px.p, pixel_values, n_px * 4, cudaMemcpyHostToDevice, cs));
  });
  return 0;
  MMEE_CATCH
}

int mmee_forward_images(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                        const int64_t* attention_mask, const mmee_images* images, const mmee_policy* policy,
                        const mmee_outputs* out) {
  MMEE_TRY
  if (!e || !out) throw std::runtime_error("null argument");
  check_images(e, B, images);
  CUDA_OK(cudaSetDevice(e->device));
  // the previous host forward has finished (it synchronises), so nothing reads img_bytes any more
  if (static_cast<int64_t>(e->img_bytes.n) < images->total_bytes) e->img_bytes.alloc(images->total_bytes);
  host_forward(e, B, input_ids, bbox, attention_mask, policy, out, [&](cudaStream_t cs) {
    CUDA_OK(cudaMemcpyAsync(e->img_bytes.p, images->data, images->total_bytes, cudaMemcpyHostToDevice, cs));
    preprocess_images(e, B, images, e->img_bytes.p, e->in_px.p, cs);
  });
  return 0;
  MMEE_CATCH
}

int mmee_preprocess_images(mmee_engine* e, int B, const mmee_images* images, float* pixel_values, void* cuda_stream) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  check_images(e, B, images);
  if (!pixel_values) throw std::runtime_error("pixel_values missing");
  CUDA_OK(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : e->stream;
  preprocess_images(e, B, images, images->data, pixel_values, st);
  if (!cuda_stream) CUDA_OK(cudaStreamSynchronize(st));
  return 0;
  MMEE_CATCH
}

int mmee_forward_submit(mmee_engine* e, int B, const int64_t* input_ids, const int64_t* bbox,
                        const int64_t* attention_mask, const float* pixel_values, const mmee_policy* policy) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  if (B < 1 || B > e->max_batch) throw std::runtime_error("batch out of range");
  CUDA_OK(cudaSetDevice(e->device));
  const int ticket = e->next_slot;
  mmee_engine::Slot& sl = e->slots[ticket];
  if (sl.busy) throw std::runtime_error("both pipeline slots are in flight: collect a ticket first");
  const int T = e->T, K = e->K, E1 = e->d.n_exits + 1;
  const size_t n_ids = static_cast<size_t>(B) * T, n_px = static_cast<size_t>(B) * e->d.channels * e->d.image * e->d.image;
  if (!sl.done) {
    const size_t mb = e->max_batch;
    sl.ids.alloc(mb * T); sl.bbox.alloc(mb * T * 4); sl.mask.alloc(mb * T);
    sl.px.alloc(mb * e->d.channels * e->d.image * e->d.image);
    sl.logits.alloc(mb * K); sl.crit.alloc(mb); sl.exit_index.alloc(mb); sl.hist.alloc(E1);
    CUDA_OK(cudaEventCreateWithFlags(&sl.small_ready, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&sl.px_ready, cudaEventDisableTiming));
    CUDA_OK(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
  }
  // all uploads on the copy stream: they overlap the forward that is still running on the compute stream
  cudaStream_t cs = e->copy_stream, st = e->stream;
  CUDA_OK(cudaMemcpyAsync(sl.ids.p, input_ids, n_ids * 8, cudaMemcpyHostToDevice, cs));
  CUDA_OK(cudaMemcpyAsync(sl.bbox.p, bbox, n_ids * 32, cudaMemcpyHostToDevice, cs));
  CUDA_OK(cudaMemcpyAsync(sl.mask.p, attention_mask, n_ids * 8, cudaMemcpyHostToDevice, cs));
  CUDA_OK(cudaEventRecord(sl.small_ready, cs));
  CUDA_OK(cudaMemcpyAsync(sl.px.p, pixel_values, n_px * 4, cudaMemcpyHostToDevice, cs));
  CUDA_OK(cudaEventRecord(sl.px_ready, cs));
  CUDA_OK(cudaStreamWaitEvent(st, sl.small_ready, 0));
  mmee_outputs dv{};
  dv.logits = e->out_logits.p; dv.exit_index = e->out_exit.p; dv.criterion = e->out_crit.p;
  dv.exit_hist = reinterpret_cast<int64_t*>(e->hist64.p);
  e->px_async = true;
  e->px_wait = sl.px_ready;
  try {
    forward_device(e, B, sl.ids.p, sl.bbox.p, sl.mask.p, sl.px.p, policy, &dv, st);
  } catch (...) {
    e->px_async = false; e->px_wait = nullptr;
    throw;
  }
  e->px_async = false; e->px_wait = nullptr;
  // stage the results: the next forward overwrites the engine's own output buffers
  CUDA_OK(cudaMemcpyAsync(sl.logits.p, e->out_logits.p, static_cast<size_t>(B) * K * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_OK(cudaMemcpyAsync(sl.exit_index.p, e->out_exit.p, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_OK(cudaMemcpyAsync(sl.crit.p, e->out_crit.p, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToDevice, st));
  CUDA_OK(cudaMemcpyAsync(sl.hist.p, e->hist64.p, static_cast<size_t>(E1) * 8, cudaMemcpyDeviceToDevice, st));
  CUDA_OK(cudaEventRecord(sl.done, st));
  sl.B = B;
  sl.busy = true;
  e->next_slot ^= 1;
  return ticket;
  MMEE_CATCH
}

int mmee_forward_collect(mmee_engine* e, int ticket, const mmee_outputs* out) {
  MMEE_TRY
  if (!e || !out || !out->logits || !out->exit_index) throw std::runtime_error("null argument");
  if (ticket < 0 || ticket > 1 || !e->slots[ticket].busy) throw std::runtime_error("no forward in flight for this ticket");
  CUDA_OK(cudaSetDevice(e->device));
  mmee_engine::Slot& sl = e->slots[ticket];
  const int B = sl.B, K = e->K, E1 = e->d.n_exits + 1;
  CUDA_OK(cudaEventSynchronize(sl.done));
  sl.busy = false;
  CUDA_OK(cudaMemcpy(out->logits, sl.logits.p, static_cast<size_t>(B) * K * 4, cudaMemcpyDeviceToHost));
  CUDA_OK(cudaMemcpy(out->exit_index, sl.exit_index.p, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost));
  if (out->criterion) CUDA_OK(cudaMemcpy(out->criterion, sl.crit.p, static_cast<size_t>(B) * 4, cudaMemcpyDeviceToHost));
  if (out->exit_hist) CUDA_OK(cudaMemcpy(out->exit_hist, sl.hist.p, static_cast<size_t>(E1) * 8, cudaMemcpyDeviceToHost));
  check_error_flags(e);
  return 0;
  MMEE_CATCH
}

int mmee_plan_create(mmee_engine* e, int B, const mmee_policy* shape, int want_all, mmee_plan** out) {
  MMEE_TRY
  if (!e || !shape || !out) throw std::runtime_error("null argument");
  if (!e->finalized) throw std::runtime_error("weights not finalized");
  if (B < 1 || B > e->max_batch) throw std::runtime_error("batch out of range");
  if (shape->criterion < 0 || shape->criterion > 2) throw std::runtime_error("criterion must be 0, 1 or 2");
  if (shape->mode != 0 && shape->mode != 1) throw std::runtime_error("mode must be 0 (dense) or 1 (early exit)");
  if (shape->criterion == MMEE_CRIT_LTE && !e->lte_w.p)
    throw std::runtime_error("criterion LTE needs the weights layoutlmv3.encoder.lte_classifier.{weight,bias}");
  CUDA_OK(cudaSetDevice(e->device));
  alloc_inputs(e);
  std::unique_ptr<mmee_plan> p(new mmee_plan());
  p->e = e; p->B = B; p->criterion = shape->criterion; p->mode = shape->mode; p->want_all = want_all != 0;
  const int E1 = e->d.n_exits + 1;
  p->policy_dev.alloc(static_cast<size_t>(2) * E1, true);
  CUDA_OK(cudaMallocHost(&p->policy_host, static_cast<size_t>(2) * E1 * sizeof(float)));
  CUDA_OK(cudaEventCreateWithFlags(&p->policy_copied, cudaEventDisableTiming));
  warm_up(e, B, p->criterion);
  capture_plan(p.get());
  CUDA_OK(cudaGraphInstantiate(&p->exec, p->graph, 0));
  CUDA_OK(cudaGraphUpload(p->exec, e->stream));
  CUDA_OK(cudaStreamSynchronize(e->stream));
  e->plans.push_back(p.get());
  *out = p.release();
  return 0;
  MMEE_CATCH
}

int mmee_plan_forward(mmee_plan* p, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                      const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out) {
  MMEE_TRY
  if (!p) throw std::runtime_error("null plan");
  mmee_engine* e = p->e;
  CUDA_OK(cudaSetDevice(e->device));
  plan_run(p, input_ids, bbox, attention_mask, pixel_values, policy, out, e->stream, true);
  CUDA_OK(cudaStreamSynchronize(e->stream));
  check_error_flags(e);
  return 0;
  MMEE_CATCH
}

int mmee_plan_forward_device(mmee_plan* p, const int64_t* input_ids, const int64_t* bbox, const int64_t* attention_mask,
                             const float* pixel_values, const mmee_policy* policy, const mmee_outputs* out,
                             void* cuda_stream) {
  MMEE_TRY
  if (!p) throw std::runtime_error("null plan");
  mmee_engine* e = p->e;
  CUDA_OK(cudaSetDevice(e->device));
  cudaStream_t st = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : e->stream;
  plan_run(p, input_ids, bbox, attention_mask, pixel_values, policy, out, st, false);
  if (!cuda_stream) {
    CUDA_OK(cudaStreamSynchronize(st));
    check_error_flags(e);
  }
  return 0;
  MMEE_CATCH
}

void mmee_plan_destroy(mmee_plan* p) {
  if (p) plan_destroy(p);
}

int64_t mmee_last_launch_count(mmee_engine* e) { return e ? e->launches : -1; }

int mmee_sync(mmee_engine* e, void* cuda_stream) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaStreamSynchronize(cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : e->stream));
  collect_profile(e);
  check_error_flags(e);
  return 0;
  MMEE_CATCH
}

int mmee_collect_profile(mmee_engine* e) {
  MMEE_TRY
  if (!e) throw std::runtime_error("null engine");
  CUDA_OK(cudaSetDevice(e->device));
  CUDA_OK(cudaDeviceSynchronize());
  collect_profile(e);
  return 0;
  MMEE_CATCH
}

int64_t mmee_debug_read(mmee_engine* e, const char* name, void* host_dst, int64_t capacity_bytes) {
  try {
    if (!e || !name || !host_dst) throw std::runtime_error("null argument");
    CUDA_OK(cudaSetDevice(e->device));
    CUDA_OK(cudaDeviceSynchronize());
    const std::string n(name);
    const void* src = nullptr;
    size_t bytes = 0;
    if (n == "X0") { src = e->X[0].p; bytes = e->X[0].n * 2; }
    else if (n == "X1") { src = e->X[1].p; bytes = e->X[1].n * 2; }
    else if (n == "QK") { src = e->QK.p; bytes = e->QK.n * 2; }
    else if (n == "VT") { src = e->VT.p; bytes = e->VT.n * 2; }
    else if (n == "CTX") { src = e->CTX.p; bytes = e->CTX.n * 2; }
    else if (n == "A1") { src = e->A1.p; bytes = e->A1.n * 2; }
    else if (n == "MID") { src = e->MID.p; bytes = e->MID.n * 2; }
    else if (n == "Y") { src = e->Y.p; bytes = e->Y.n * 4; }
    else if (n == "Y2") { src = e->Y2.p; bytes = e->Y2.n * 4; }
    else if (n == "VIS") { src = e->VIS.p; bytes = e->VIS.n * 4; }
    else if (n == "POOL") { src = e->POOL.p; bytes = e->POOL.n * 4; }
    else if (n == "ATT_TRACE") { src = e->att_trace.p; bytes = e->att_trace.n * 8; }
    else if (n == "BIAS") { src = e->BIAS.p; bytes = e->BIAS.n * 2; }
    else if (n == "BIASlo") { src = e->BIASlo.p; bytes = e->BIASlo.n * 2; }
    else if (n == "X0lo") { src = e->Xlo[0].p; bytes = e->Xlo[0].n * 2; }
    else if (n == "QKlo") { src = e->QKlo.p; bytes = e->QKlo.n * 2; }
    else if (n == "CTXlo") { src = e->CTXlo.p; bytes = e->CTXlo.n * 2; }
    else if (n == "MIDlo") { src = e->MIDlo.p; bytes = e->MIDlo.n * 2; }
    else if (n == "NDEV") { src = e->n_dev.p; bytes = e->n_dev.n * 4; }
    else throw std::runtime_error("unknown buffer " + n);
    if (static_cast<int64_t>(bytes) > capacity_bytes) bytes = static_cast<size_t>(capacity_bytes);
    CUDA_OK(cudaMemcpy(host_dst, src, bytes, cudaMemcpyDeviceToHost));
    return static_cast<int64_t>(bytes);
  } catch (const std::exception& ex) {
    g_err = ex.what();
    return -1;
  }
}

}  // extern "C"

// Device-resident store of per-exit criteria (SURVEY.md §8 f2): the logits go up once, every sweep after that only
// moves thresholds in and histograms out.
struct mmee_policy_store {
  int device = 0, E1 = 0, K = 0, criterion = 0;
  int64_t N = 0;
  bool has_labels = false;
  DevBuf<double> crit;
  DevBuf<int> argmax;
  DevBuf<int64_t> labels;
  DevBuf<unsigned long long> cmask;
};

namespace {

template <int NE>
void launch_policy_hist(bool strict, unsigned blocks, size_t smem, const mmee_policy_store* ps, const double* thr,
                        int64_t n_thr, int cmp, int n_test, int fallback, long long* hist, long long* correct) {
  const unsigned long long* cm = ps->has_labels ? ps->cmask.p : nullptr;
  // [chunk][E1 + 1] doubles of staged criteria: above the 48 KB default from E1 = 24 on
  CUDA_OK(cudaFuncSetAttribute(policy_hist_kernel<NE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  CUDA_OK(cudaFuncSetAttribute(policy_hist_kernel<NE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  if (strict)
    policy_hist_kernel<NE, true><<<blocks, POLICY_HIST_THREADS, smem>>>(ps->crit.p, cm, thr, ps->E1, ps->N, n_thr, cmp,
                                                                        n_test, fallback, hist, correct);
  else
    policy_hist_kernel<NE, false><<<blocks, POLICY_HIST_THREADS, smem>>>(ps->crit.p, cm, thr, ps->E1, ps->N, n_thr, cmp,
                                                                         n_test, fallback, hist, correct);
}

void policy_store_scan(mmee_policy_store* ps, const double* thresholds, int64_t n_thr, int mode, int32_t* exits_out,
                       int64_t* hist_out, int64_t* correct_out) {
  if (!ps || !thresholds) throw std::runtime_error("null argument");
  if (n_thr < 1) throw std::runtime_error("bad shape");
  if (mode != 0 && mode != 1) throw std::runtime_error("mode must be 0 (policy.py) or 1 (check_2D_threshold)");
  if (correct_out && !ps->has_labels) throw std::runtime_error("correct_out needs a store created with labels");
  CUDA_OK(cudaSetDevice(ps->device));
  const int E1 = ps->E1;
  const int64_t N = ps->N;
  // mode 0: EE/policy.py:28-45 (strict, last exit unconditional); mode 1: EE/thresh.py:184-185 (>=, every exit
  // tested, nothing fired -> exit 0; the entropy CSF is the negated entropy, EE/large_scale.py:15)
  // larger = more confident for max softmax and margin, smaller for entropy
  const int cmp = mode == 0 ? (ps->criterion == 1 ? POLICY_LT : POLICY_GT) : (ps->criterion == 1 ? POLICY_LE : POLICY_GE);
  const int n_test = mode == 0 ? E1 - 1 : E1;
  const int fallback = mode == 0 ? E1 - 1 : 0;
  std::vector<double> neg;
  if (mode == 1 && ps->criterion == 1) {            // -H >= thr  <=>  H <= -thr
    neg.assign(thresholds, thresholds + static_cast<size_t>(n_thr) * E1);
    for (auto& v : neg) v = -v;
    thresholds = neg.data();
  }
  DevBuf<double> d_thr;
  d_thr.alloc(static_cast<size_t>(n_thr) * E1);
  CUDA_OK(cudaMemcpy(d_thr.p, thresholds, static_cast<size_t>(n_thr) * E1 * 8, cudaMemcpyHostToDevice));
  const bool by_threshold = !exits_out && E1 <= 64 && n_thr >= 2048;
  if (by_threshold) {
    // thread = sweep point: no [n_thr, N] index matrix, no atomics (policy_hist_kernel)
    DevBuf<long long> d_hist, d_correct;
    d_hist.alloc(static_cast<size_t>(n_thr) * E1);
    if (correct_out) d_correct.alloc(n_thr);
    const unsigned blocks = static_cast<unsigned>((n_thr + POLICY_HIST_THREADS - 1) / POLICY_HIST_THREADS);
    const size_t smem = static_cast<size_t>(POLICY_HIST_CHUNK) * (E1 + 1) * 8;
    const bool strict = mode == 0;
    if (E1 <= 8) launch_policy_hist<8>(strict, blocks, smem, ps, d_thr.p, n_thr, cmp, n_test, fallback, d_hist.p, d_correct.p);
    else if (E1 <= 16) launch_policy_hist<16>(strict, blocks, smem, ps, d_thr.p, n_thr, cmp, n_test, fallback, d_hist.p, d_correct.p);
    else if (E1 <= 32) launch_policy_hist<32>(strict, blocks, smem, ps, d_thr.p, n_thr, cmp, n_test, fallback, d_hist.p, d_correct.p);
    else launch_policy_hist<64>(strict, blocks, smem, ps, d_thr.p, n_thr, cmp, n_test, fallback, d_hist.p, d_correct.p);
    CUDA_OK(cudaGetLastError());
    if (hist_out) CUDA_OK(cudaMemcpy(hist_out, d_hist.p, static_cast<size_t>(n_thr) * E1 * 8, cudaMemcpyDeviceToHost));
    if (correct_out) CUDA_OK(cudaMemcpy(correct_out, d_correct.p, static_cast<size_t>(n_thr) * 8, cudaMemcpyDeviceToHost));
    CUDA_OK(cudaDeviceSynchronize());
    return;
  }
  // thread = sample, sweep points along grid.y in chunks of <= 65535 (the grid limit)
  DevBuf<int32_t> d_exits;
  DevBuf<unsigned long long> d_hist, d_correct;
  const int64_t chunk_max = 65535;
  const int64_t rows_buf = std::min<int64_t>(n_thr, chunk_max);
  if (exits_out) d_exits.alloc(static_cast<size_t>(rows_buf) * N);
  d_hist.alloc(static_cast<size_t>(n_thr) * E1, true);
  d_correct.alloc(n_thr, true);
  for (int64_t t0 = 0; t0 < n_thr; t0 += chunk_max) {
    const int64_t nt = std::min<int64_t>(chunk_max, n_thr - t0);
    policy_scan_kernel<<<dim3(static_cast<unsigned>((N + 255) / 256), static_cast<unsigned>(nt)), 256,
                         (E1 + 1) * sizeof(unsigned int)>>>(
        ps->crit.p, ps->argmax.p, d_thr.p + static_cast<size_t>(t0) * E1, ps->has_labels ? ps->labels.p : nullptr, E1, N, cmp,
        n_test, fallback, exits_out ? d_exits.p : nullptr, d_hist.p + static_cast<size_t>(t0) * E1, d_correct.p + t0);
    CUDA_OK(cudaGetLastError());
    if (exits_out)
      CUDA_OK(cudaMemcpy(exits_out + static_cast<size_t>(t0) * N, d_exits.p, static_cast<size_t>(nt) * N * 4, cudaMemcpyDeviceToHost));
  }
  if (hist_out) CUDA_OK(cudaMemcpy(hist_out, d_hist.p, static_cast<size_t>(n_thr) * E1 * 8, cudaMemcpyDeviceToHost));
  if (correct_out) CUDA_OK(cudaMemcpy(correct_out, d_correct.p, static_cast<size_t>(n_thr) * 8, cudaMemcpyDeviceToHost));
  CUDA_OK(cudaDeviceSynchronize());
}

mmee_policy_store* policy_store_create(int device, int E1, int64_t N, int K, const double* logits, const double* temperatures,
                                       int criterion, const int64_t* labels) {
  if (!logits) throw std::runtime_error("null argument");
  if (E1 < 1 || N < 1 || K < 1) throw std::runtime_error("bad shape");
  if (criterion < 0 || criterion > 2) throw std::runtime_error("criterion must be 0 (max_confidence), 1 (entropy) or 2 (margin)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    throw std::runtime_error("no CUDA device: libmmee has no CPU fallback");
  CUDA_OK(cudaSetDevice(device));
  std::unique_ptr<mmee_policy_store> ps(new mmee_policy_store());
  ps->device = device; ps->E1 = E1; ps->N = N; ps->K = K; ps->criterion = criterion;
  const size_t n_log = static_cast<size_t>(E1) * N * K, n_en = static_cast<size_t>(E1) * N;
  DevBuf<double> d_logits, d_temps;
  d_logits.alloc(n_log);
  ps->crit.alloc(n_en);
  ps->argmax.alloc(n_en);
  CUDA_OK(cudaMemcpy(d_logits.p, logits, n_log * 8, cudaMemcpyHostToDevice));
  if (temperatures) {
    d_temps.alloc(E1);
    CUDA_OK(cudaMemcpy(d_temps.p, temperatures, static_cast<size_t>(E1) * 8, cudaMemcpyHostToDevice));
  }
  policy_crit_kernel<<<static_cast<unsigned>((n_en + 255) / 256), 256>>>(d_logits.p, d_temps.p, E1, N, K, criterion,
                                                                          ps->crit.p, ps->argmax.p);
  CUDA_OK(cudaGetLastError());
  if (labels) {
    ps->has_labels = true;
    ps->labels.alloc(N);
    ps->cmask.alloc(N);
    CUDA_OK(cudaMemcpy(ps->labels.p, labels, static_cast<size_t>(N) * 8, cudaMemcpyHostToDevice));
    policy_cmask_kernel<<<static_cast<unsigned>((N + 255) / 256), 256>>>(ps->argmax.p, ps->labels.p, E1, N, ps->cmask.p);
    CUDA_OK(cudaGetLastError());
  }
  CUDA_OK(cudaDeviceSynchronize());
  return ps.release();
}

}  // namespace

extern "C" {

int mmee_policy_store_create(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                             const double* temperatures, int criterion, const int64_t* labels, mmee_policy_store** out) {
  MMEE_TRY
  if (!out) throw std::runtime_error("null argument");
  *out = policy_store_create(device, n_exits_plus1, n_samples, n_labels, logits, temperatures, criterion, labels);
  return 0;
  MMEE_CATCH
}

void mmee_policy_store_destroy(mmee_policy_store* ps) {
  if (!ps) return;
  cudaSetDevice(ps->device);
  delete ps;
}

int mmee_policy_store_criteria(mmee_policy_store* ps, double* crit_out) {
  MMEE_TRY
  if (!ps || !crit_out) throw std::runtime_error("null argument");
  CUDA_OK(cudaSetDevice(ps->device));
  CUDA_OK(cudaMemcpy(crit_out, ps->crit.p, static_cast<size_t>(ps->E1) * ps->N * 8, cudaMemcpyDeviceToHost));
  return 0;
  MMEE_CATCH
}

int mmee_policy_store_scan(mmee_policy_store* ps, const double* thresholds, int64_t n_thr, int mode, int32_t* exits_out,
                           int64_t* hist_out, int64_t* correct_out) {
  MMEE_TRY
  policy_store_scan(ps, thresholds, n_thr, mode, exits_out, hist_out, correct_out);
  return 0;
  MMEE_CATCH
}

int mmee_policy_scan(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                     const double* temperatures, int criterion, const double* thresholds, int n_thr,
                     const int64_t* labels, int32_t* exits_out, double* crit_out, int64_t* hist_out,
                     int64_t* correct_out) {
  MMEE_TRY
  if (!thresholds) throw std::runtime_error("null argument");
  std::unique_ptr<mmee_policy_store> ps(
      policy_store_create(device, n_exits_plus1, n_samples, n_labels, logits, temperatures, criterion, labels));
  policy_store_scan(ps.get(), thresholds, n_thr, 0, exits_out, hist_out, labels ? correct_out : nullptr);
  if (crit_out)
    CUDA_OK(cudaMemcpy(crit_out, ps->crit.p, static_cast<size_t>(ps->E1) * ps->N * 8, cudaMemcpyDeviceToHost));
  return 0;
  MMEE_CATCH
}

}  // extern "C"

namespace {
// shared body of mmee_temperature_fit / mmee_calibration_stats: logits + labels to the device, `iters` Newton
// iterations from t_init (0: none), then one statistics pass at the final temperatures
void calibration_run(int device, int E1, int64_t N, int K, const double* logits, const int64_t* labels,
                     const double* t_init, int iters, double* t_out, double* nll_before, double* nll_out,
                     double* conf_out, double* acc_out) {
  if (!logits || !labels) throw std::runtime_error("null argument");
  if (E1 < 1 || N < 1 || K < 1) throw std::runtime_error("bad shape");
  for (int64_t i = 0; i < N; ++i)
    if (labels[i] < 0 || labels[i] >= K) throw std::runtime_error("label out of range");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    throw std::runtime_error("no CUDA device: libmmee has no CPU fallback");
  CUDA_OK(cudaSetDevice(device));
  const size_t n_log = static_cast<size_t>(E1) * N * K;
  const int blocks = static_cast<int>(std::min<int64_t>((N + CALIB_THREADS - 1) / CALIB_THREADS, 64));
  DevBuf<double> d_logits, d_beta, d_partial, d_stats;
  DevBuf<int64_t> d_labels;
  DevBuf<CalibState> d_state;
  d_logits.alloc(n_log); d_labels.alloc(N); d_beta.alloc(E1);
  d_partial.alloc(static_cast<size_t>(E1) * blocks * CALIB_NSTAT); d_stats.alloc(static_cast<size_t>(E1) * CALIB_NSTAT);
  d_state.alloc(E1);
  std::vector<double> beta(E1);
  std::vector<CalibState> st(E1);
  for (int e = 0; e < E1; ++e) {
    const double t = t_init ? t_init[e] : 1.0;
    if (!(t > 0.0)) throw std::runtime_error("temperatures must be positive");
    beta[e] = 1.0 / t;
    st[e] = CalibState{beta[e], beta[e], 0.0, 0.0, 0.0, 0};
  }
  CUDA_OK(cudaMemcpy(d_logits.p, logits, n_log * 8, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d_labels.p, labels, static_cast<size_t>(N) * 8, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d_beta.p, beta.data(), static_cast<size_t>(E1) * 8, cudaMemcpyHostToDevice));
  CUDA_OK(cudaMemcpy(d_state.p, st.data(), static_cast<size_t>(E1) * sizeof(CalibState), cudaMemcpyHostToDevice));
  const unsigned ub = (E1 + 31) / 32;
  for (int it = 0; it < iters; ++it) {
    calib_stats_kernel<<<dim3(blocks, E1), CALIB_THREADS>>>(d_logits.p, d_labels.p, d_beta.p, N, K, d_partial.p);
    calib_update_kernel<<<ub, 32>>>(d_partial.p, blocks, N, E1, d_state.p, d_beta.p, d_stats.p, 1);
  }
  CUDA_OK(cudaGetLastError());
  if (iters > 0) {
    // the last ACCEPTED point is the answer (the pending trial step is dropped)
    CUDA_OK(cudaMemcpy(st.data(), d_state.p, static_cast<size_t>(E1) * sizeof(CalibState), cudaMemcpyDeviceToHost));
    for (int e = 0; e < E1; ++e) beta[e] = st[e].beta_ok;
    CUDA_OK(cudaMemcpy(d_beta.p, beta.data(), static_cast<size_t>(E1) * 8, cudaMemcpyHostToDevice));
  }
  calib_stats_kernel<<<dim3(blocks, E1), CALIB_THREADS>>>(d_logits.p, d_labels.p, d_beta.p, N, K, d_partial.p);
  calib_update_kernel<<<ub, 32>>>(d_partial.p, blocks, N, E1, d_state.p, d_beta.p, d_stats.p, 0);
  CUDA_OK(cudaGetLastError());
  std::vector<double> stats(static_cast<size_t>(E1) * CALIB_NSTAT);
  CUDA_OK(cudaMemcpy(stats.data(), d_stats.p, stats.size() * 8, cudaMemcpyDeviceToHost));
  for (int e = 0; e < E1; ++e) {
    if (t_out) t_out[e] = 1.0 / beta[e];
    if (nll_before) nll_before[e] = iters > 0 ? st[e].nll_first : stats[e * CALIB_NSTAT + 0];
    if (nll_out) nll_out[e] = stats[e * CALIB_NSTAT + 0];
    if (conf_out) conf_out[e] = stats[e * CALIB_NSTAT + 3];
    if (acc_out) acc_out[e] = stats[e * CALIB_NSTAT + 4];
  }
}
}  // namespace

extern "C" {

int mmee_temperature_fit(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                         const int64_t* labels, const double* t_init, int max_iter, double* t_out, double* nll_before,
                         double* nll_after, double* mean_conf_out, double* accuracy_out) {
  MMEE_TRY
  if (!t_out) throw std::runtime_error("null argument");
  calibration_run(device, n_exits_plus1, n_samples, n_labels, logits, labels, t_init, max_iter > 0 ? max_iter : 40,
                  t_out, nll_before, nll_after, mean_conf_out, accuracy_out);
  return 0;
  MMEE_CATCH
}

int mmee_calibration_stats(int device, int n_exits_plus1, int64_t n_samples, int n_labels, const double* logits,
                           const int64_t* labels, const double* temperatures, double* nll_out, double* mean_conf_out,
                           double* accuracy_out) {
  MMEE_TRY
  calibration_run(device, n_exits_plus1, n_samples, n_labels, logits, labels, temperatures, 0, nullptr, nullptr,
                  nll_out, mean_conf_out, accuracy_out);
  return 0;
  MMEE_CATCH
}

int mmee_set_profiling(mmee_engine* e, int on) {
  if (!e) return -1;
  for (auto& x : e->ev) cudaEventDestroy(x.second);    // (re)start the accumulation
  e->ev.clear();
  e->stage_ms.clear();
  e->profiling = (on & 1) != 0;
  e->trace_on = (on & 2) != 0;     // developer trace of the first layer's attention kernel (debug_read "ATT_TRACE")
  return 0;
}

double mmee_last_stage_ms(mmee_engine* e, const char* stage) {
  if (!e || !stage) return -1.0;
  auto it = e->stage_ms.find(stage);
  return it == e->stage_ms.end() ? 0.0 : it->second;
}

}  // extern "C"
