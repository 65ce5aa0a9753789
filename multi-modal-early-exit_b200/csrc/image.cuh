// Device preprocess of uint8 document images (mmee_preprocess_images, mmee_forward_images): what the reference's
// LayoutLMv3 image processor gives for Image.fromarray(page).convert("RGB"), bit for bit (oracle/image_port.py):
//   Pillow's Image.resize((S, S), BILINEAR) on 8-bit data, then (r / 255 - 0.5) / 0.5 in fp32, into [3, S, S].
//   image_coeffs_kernel : Pillow's fixed-point bilinear coefficients (Resample.c precompute_coeffs +
//                         normalize_coeffs_8bpc), one CTA per distinct input length of an axis
//   image_pass1_kernel  : the first pass into a uint8 intermediate (horizontal; vertical for a page Pillow shrinks
//                         vertically first: more than 100 times taller than wide)
//   image_pass2_kernel  : the other pass, fused with rescale / normalise; writes fp32 [B, 3, S, S] and replicates a
//                         grayscale channel, as convert("RGB") does
// The batch is ragged: each image has its own (h, w) and byte offset.  A pass over an axis that already has S entries
// is not skipped: its coefficients are exactly {2^22, 0}, the identity.
#pragma once
#include <stdint.h>

namespace mmee {

constexpr int IMG_PRECISION_BITS = 22;   // Pillow's PRECISION_BITS for 8-bit resampling
constexpr int IMG_MAX_SIDE = 16384;

struct ImageAxis {        // one coefficient table: in_size -> S; kk[kk_off + o * ksize + x], bounds[table * S + o]
  int in_size, ksize;
  int64_t kk_off;
};

struct ImageDesc {
  int64_t src_off;        // byte offset of the image in the packed batch (row-major HWC)
  int64_t tmp_off;        // byte offset of its first-pass output in the intermediate
  int h, w;
  int th, tw;             // coefficient tables of the vertical (height) and horizontal (width) axis
  int vfirst;             // first pass is vertical: the intermediate is [S, w, C], else [h, S, C]
  int pad_;
};

// Pillow's precompute_coeffs for the bilinear filter (support 1), in fp64 with every operation rounded on its own:
// a fused multiply-add would change the coefficients.
__global__ void image_coeffs_kernel(const ImageAxis* __restrict__ axes, int S, int2* __restrict__ bounds,
                                    int* __restrict__ kk) {
  const ImageAxis ax = axes[blockIdx.x];
  const double scale = __ddiv_rn(static_cast<double>(ax.in_size), static_cast<double>(S));
  const double fs = scale < 1.0 ? 1.0 : scale;    // filterscale; support = 1.0 * filterscale
  const double support = fs;
  const double ss = __ddiv_rn(1.0, fs);
  for (int o = threadIdx.x; o < S; o += blockDim.x) {
    const double center = __dmul_rn(__dadd_rn(static_cast<double>(o), 0.5), scale);
    const int xmin = max(__double2int_rz(__dadd_rn(__dsub_rn(center, support), 0.5)), 0);
    const int xmax = min(__double2int_rz(__dadd_rn(__dadd_rn(center, support), 0.5)), ax.in_size);
    const int n = min(xmax - xmin, ax.ksize);
    auto tri = [&](int x) {
      const double t = fabs(__dmul_rn(__dadd_rn(__dsub_rn(static_cast<double>(x + xmin), center), 0.5), ss));
      return t < 1.0 ? __dsub_rn(1.0, t) : 0.0;
    };
    double ww = 0.0;
    for (int x = 0; x < n; ++x) ww = __dadd_rn(ww, tri(x));
    int* k = kk + ax.kk_off + static_cast<int64_t>(o) * ax.ksize;
    for (int x = 0; x < ax.ksize; ++x) {
      double w = x < n ? tri(x) : 0.0;
      if (ww != 0.0) w = __ddiv_rn(w, ww);
      const double sw = __dmul_rn(w, static_cast<double>(1 << IMG_PRECISION_BITS));
      k[x] = __double2int_rz(w < 0.0 ? __dadd_rn(-0.5, sw) : __dadd_rn(0.5, sw));
    }
    bounds[blockIdx.x * S + o] = make_int2(xmin, n);
  }
}

__device__ __forceinline__ uint8_t image_clip8(int ss) {
  const int v = ss >> IMG_PRECISION_BITS;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// One output element of a pass, all C channels: clip8(2^21 + sum_x p[x * step + ch] * k[x]).  Offsets inside one
// image fit in 32 bits: at most 16384 * 16384 * 3 bytes.
template <int C>
__device__ __forceinline__ void image_taps(const uint8_t* __restrict__ p, int step, const int* __restrict__ k, int n,
                                           int (&acc)[C]) {
#pragma unroll
  for (int ch = 0; ch < C; ++ch) acc[ch] = 1 << (IMG_PRECISION_BITS - 1);
#pragma unroll 1
  for (int x = 0; x < n; ++x) {
    const int kx = __ldg(k + x);
#pragma unroll
    for (int ch = 0; ch < C; ++ch) acc[ch] += static_cast<int>(__ldg(p + x * step + ch)) * kx;
  }
}

// grid (x: elements of one image, grid-stride; y: images, stride gridDim.y)
template <int C>
__global__ void __launch_bounds__(256, C == 1 ? 8 : 6) image_pass1_kernel(const uint8_t* __restrict__ src,
                                                             const ImageDesc* __restrict__ imgs, int B, int S,
                                                             const ImageAxis* __restrict__ axes,
                                                             const int2* __restrict__ bounds,
                                                             const int* __restrict__ kk, uint8_t* __restrict__ tmp) {
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const ImageDesc im = imgs[b];
    const bool vf = im.vfirst != 0;
    const int cols = vf ? im.w : S, n_items = (vf ? S : im.h) * cols;
    const int t = vf ? im.th : im.tw;
    const ImageAxis ax = axes[t];
    const int pitch = im.w * C;
    const uint8_t* in = src + im.src_off;
    const int* kt = kk + ax.kk_off;
    const int2* bt = bounds + t * S;
    uint8_t* q = tmp + im.tmp_off;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
      const int r = i / cols, c = i - r * cols;
      const int o = vf ? r : c;                     // output index along the resampled axis
      const int2 bd = __ldg(bt + o);
      int acc[C];
      image_taps<C>(in + (vf ? bd.x * pitch + c * C : r * pitch + bd.x * C), vf ? pitch : C, kt + o * ax.ksize, bd.y,
                    acc);
#pragma unroll
      for (int ch = 0; ch < C; ++ch) q[i * C + ch] = image_clip8(acc[ch]);
    }
  }
}

// grid as image_pass1_kernel.  Rescale + normalise through a table of the 256 byte values: (r / 255 - 0.5) / 0.5 in
// IEEE fp32 with correctly rounded division (LayoutLMv3 mean = std = 0.5).
template <int C>
__global__ void __launch_bounds__(256, 8) image_pass2_kernel(const uint8_t* __restrict__ tmp,
                                                             const ImageDesc* __restrict__ imgs, int B, int S,
                                                             const ImageAxis* __restrict__ axes,
                                                             const int2* __restrict__ bounds,
                                                             const int* __restrict__ kk, float* __restrict__ out) {
  __shared__ float norm[256];
  for (int r = threadIdx.x; r < 256; r += blockDim.x)
    norm[r] = __fdiv_rn(__fsub_rn(__fdiv_rn(static_cast<float>(r), 255.0f), 0.5f), 0.5f);
  __syncthreads();
  const int n_items = S * S;
  for (int b = blockIdx.y; b < B; b += gridDim.y) {
    const ImageDesc im = imgs[b];
    const bool vf = im.vfirst != 0;
    const int cols = vf ? im.w : S;                 // columns of the intermediate
    const int t = vf ? im.tw : im.th;
    const ImageAxis ax = axes[t];
    const int pitch = cols * C;
    const uint8_t* in = tmp + im.tmp_off;
    const int* kt = kk + ax.kk_off;
    const int2* bt = bounds + t * S;
    float* ob = out + static_cast<int64_t>(b) * 3 * n_items;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_items; i += gridDim.x * blockDim.x) {
      const int yy = i / S, xx = i - yy * S;
      const int o = vf ? xx : yy;
      const int2 bd = __ldg(bt + o);
      int acc[C];
      image_taps<C>(in + (vf ? yy * pitch + bd.x * C : bd.x * pitch + xx * C), vf ? C : pitch, kt + o * ax.ksize,
                    bd.y, acc);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) ob[ch * n_items + i] = norm[image_clip8(acc[C == 1 ? 0 : ch])];
    }
  }
}

}  // namespace mmee
